/*
 * seriation_b200.h -- C ABI of the B200-native seriation MCMC sweep.
 *
 * This is the drop-in boundary for ONE path of the reference
 * (PrayagS/Seriation-in-Paleontological-Data-using-MCMC): the per-chain sweep of
 * C_Implementation/mcmc.c and the cross-chain selection / pair-order steps of
 * script.py.  Plain C types only; every entry point returns 0 on success or a
 * negative SER_E_* code, and ser_last_error() describes the failure.  The
 * library is CUDA-only: without a usable device every compute entry point fails
 * with SER_E_CUDA -- there is no CPU fallback.
 *
 * Reference interfaces replaced (file:line under /root/reference):
 *   ser_dataset_read_txt      mcmc_readmodel            C_Implementation/mcmc.c:339-401
 *   ser_dataset_read_names    (.genus/.sites files)     Dataset/g*.genus, Dataset/g*.sites
 *   ser_run_create/_init      mcmc_init+mcmc_randomize  mcmc.c:581-593, :477-578, :440-474
 *   ser_run_advance           mcmc_sample loop          mcmc.c:214-258 (main: :140-143, :180-185)
 *   ser_run_get_state         mcmc_model fields         mcmc.h:32-45
 *   ser_run_fetch_samples     mcmc_save_chain rows      mcmc.c:69-92
 *   ser_run_get_cd/_fetch_cd_samples  per-taxon c[], d[] (manycd)  mcmc.c:777-785, :807-815, :82-91
 *   ser_run_chain_stats       compute/print_exp_data    mcmc.c:53-67
 *   ser_run_check             mcmc_consistent           mcmc.c:999-1094
 *   ser_write_chain_files     main's five fopen()s      mcmc.c:148-197, :261-294
 *   ser_select_chains*        choose_chains             script.py:70-99
 *   ser_run_po_counts*        compute_pair_order_matrix script.py:155-189
 *   ser_run_posterior_sums    compute_exp_ages / compute_exp_pi / compute_exp_a
 *                                                       script.py:129-152, :230-276
 *   ser_run_alive_counts      plot_taxa_occurence_probability_matrix / plot_false_*  script.py:306-448
 *   ser_run_site_age_corr     CORR_MN of Docs/Report.pdf Table 1 (E[pi] against the .sites MN ages)
 *   run_all_chains' Pool(8) over 100 processes (script.py:48-67) is replaced by
 *   n_chains in ser_run_config: one persistent launch over all chains of a GPU, and by
 *   ser_multi_* / ser_comm_*: the chains of one call sharded over the GPUs of a box.
 */
#ifndef SERIATION_B200_H
#define SERIATION_B200_H

#include <stddef.h>
#include <stdint.h>
#include <stdio.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SER_OK 0
#define SER_E_ARG (-1)    /* bad argument / unsupported shape */
#define SER_E_PARSE (-2)  /* dataset parse error (mcmc_readmodel's exit(1) cases) */
#define SER_E_CUDA (-3)   /* CUDA runtime error or no device */
#define SER_E_STATE (-4)  /* call order (e.g. advance before init) */
#define SER_E_IO (-5)     /* file I/O */
#define SER_E_TAPE (-6)   /* replay tape missing / exhausted */
#define SER_E_CHECK (-7)  /* consistency check failed */

#define SER_MODE_FREE 0   /* counter-based Philox stream keyed by (seed, global chain id) */
#define SER_MODE_REPLAY 1 /* consume recorded draw tapes (grammar: DESIGN.md / oracle/draw_source.h) */

#define SER_STORE_NONE 0  /* per-chain running sums only */
#define SER_STORE_PI 1    /* + pi of every thinned sample (enough for the pair-order matrix) */
#define SER_STORE_FULL 2  /* + a, b, c, d, loglik of every thinned sample (chain_data.csv) */

/* limits of this build (DESIGN.md "shapes") */
#define SER_MAX_SITES 2048
#define SER_MAX_TAXA 8192

typedef struct ser_dataset ser_dataset;
typedef struct ser_run ser_run;

typedef struct ser_run_config {
  uint32_t struct_size;    /* = sizeof(ser_run_config): ser_run_create refuses a caller built against another layout */
  int32_t n_chains;        /* chains simulated by THIS process / device                        */
  int32_t chain_offset;    /* global id of local chain 0 (sharding across ranks)              */
  int32_t sweeps_per_call; /* sweeps per thinned sample; the reference hard-codes 10           */
  int32_t mode;            /* SER_MODE_*                                                       */
  uint32_t seed;           /* free-running stream seed (GSL_RNG_SEED's role)                   */
  int32_t store;           /* SER_STORE_*                                                      */
  int32_t max_samples;     /* capacity of the thinned-sample store per chain                   */
  int32_t device;          /* CUDA device ordinal                                              */
  int32_t manycd;          /* 1: per-taxon c, d (mcmc_readmodel's manycd, mcmc.c:363, :777-785); any supported shape */
} ser_run_config;

const char *ser_last_error(void);
const char *ser_version(void);

/* ---------------------------------------------------------------- datasets (host only) */
/* X: N*M row-major bytes (row = site, column = taxon, non-zero = present); hard: N flags or NULL */
int ser_dataset_from_bits(int32_t N, int32_t M, const uint8_t *X, const uint8_t *hard, ser_dataset **out);
/* the reference's .txt format; path == NULL reads stdin */
int ser_dataset_read_txt(const char *path, ser_dataset **out);
int ser_dataset_read_stream(FILE *f, ser_dataset **out);
int ser_dataset_dims(const ser_dataset *ds, int32_t *N, int32_t *M, int32_t *nh);
int ser_dataset_get(const ser_dataset *ds, uint8_t *X, uint8_t *hard);
void ser_dataset_free(ser_dataset *ds);
/* .genus (one taxon name per line) / .sites ("Name [MN,age]" + optional " *") readers.
 * Attaches labels to the dataset; counts must match M / N. */
int ser_dataset_read_names(ser_dataset *ds, const char *genus_path, const char *sites_path);
const char *ser_dataset_taxon_name(const ser_dataset *ds, int32_t m);
const char *ser_dataset_site_name(const ser_dataset *ds, int32_t n);
int ser_dataset_site_age(const ser_dataset *ds, int32_t n, int32_t *mn_unit, double *age_ma, int32_t *hard);
/* deterministic synthetic occurrence matrix (BASELINE.json config 5; generator in DESIGN.md) */
int ser_dataset_synthetic(int32_t N, int32_t M, int32_t n_hard, uint64_t seed, ser_dataset **out);

/* ---------------------------------------------------------------- runs (device) */
int ser_run_create(const ser_dataset *ds, const ser_run_config *cfg, ser_run **out);
/* A run whose local chain c is GLOBAL chain chain_ids[c] (distinct, >= 0, any order; cfg->n_chains == n, cfg->chain_offset == 0):
 * free-running chains are keyed by (seed, global id), so the chosen chains of an earlier run are re-simulated alone, bit-identical
 * to their first run (replay mode: one tape per local chain, as ever).  The cross-chain getters take global ids; local-index
 * entry points (ser_run_get_state, ser_write_chain_files, ...) keep indexing local chains.  The arguments are checked before
 * any CUDA call. */
int ser_run_create_chains(const ser_dataset *ds, const ser_run_config *cfg, const int32_t *chain_ids, int32_t n, ser_run **out);
void ser_run_destroy(ser_run *run);
/* replay mode: all chains' tapes concatenated; offsets has n_chains+1 entries (in doubles) */
int ser_run_set_tapes(ser_run *run, const double *flat, const uint64_t *offsets);
/* randomised start (mcmc_randomize) + a/b from the data + counts + log-likelihood */
int ser_run_init(ser_run *run);
/* n_calls x sweeps_per_call sweeps on every chain; if `sampling` a thinned sample is emitted
 * (and the exp_data sums advanced) after every call.  Asynchronous on the run's stream. */
int ser_run_advance(ser_run *run, int32_t n_calls, int32_t sampling);
/* burn-in calls followed by sampling calls in ONE launch (main's two loops, mcmc.c:140-143 + :180-185):
 * the persistent grid balances (chain, call) work items over the SMs across both phases */
int ser_run_advance_both(ser_run *run, int32_t burn_calls, int32_t sample_calls);
int ser_run_sync(ser_run *run);
/* CUDA-event time of all kernels launched by this run since creation / last reset, in ms */
int ser_run_elapsed_ms(ser_run *run, double *ms, int32_t reset);
int ser_run_kernel_launches(const ser_run *run, int64_t *n);
/* which sweep kernel serves this run's shape: 0 = one thread per taxon (ser_sweep_kernel), 1 = large-shape kernel with
 * CTA-wide column groups, 2 = large-shape kernel with warp batches */
int ser_run_kernel_path(const ser_run *run, int32_t *path);
/* The warp batches the large-shape kernel's Gibbs phase would use for a matrix whose sorted columns hold ones_sorted[c] ones, with
 * slices of `wcap` items per warp (host only; no device needed): batches[4 b ..] = {first column, columns | lane shift << 16,
 * first item, last item + 1}; batches may be NULL to only count them. */
int ser_plan_warp_batches(const int32_t *ones_sorted, int32_t M, int32_t wcap, int32_t *batches, int32_t max_batches, int32_t *n_batches);
/* CUDA-event time of the SWEEP launches alone since the last reset, and how many there were.  The events are
 * recorded around every launch and only read here, so measuring the dominant kernel puts no host
 * synchronisation between the launches of a timed region. */
int ser_run_sweep_time(ser_run *run, double *ms, int32_t *n_launches, int32_t reset);

/* full model state of one local chain (any pointer may be NULL) */
int ser_run_get_state(ser_run *run, int32_t chain, int32_t *a, int32_t *b, int32_t *pi, int32_t *rpi,
                      int32_t *t0, int32_t *f0, int32_t *t1, int32_t *f1, int32_t tot[4],
                      double cdl[3], int64_t *tape_slots);
/* acceptance counters of one chain: c, d, ab(changed), pi1, pi2(0), pi2(swap), pi3, sweeps */
int ser_run_get_counters(ser_run *run, int32_t chain, int64_t out[8]);
/* mcmc_consistent on every local chain, on device; *n_bad = number of inconsistent chains */
int ser_run_check(ser_run *run, int32_t *n_bad);
/* what ser_run_check found for one chain: bit 1 tape exhausted, 2 a/b out of range, 4 pi not a permutation,
 * 8 hard sites out of order, 16 totals / log-likelihood do not match a recount (mcmc.c:999-1094) */
int ser_run_get_flags(ser_run *run, int32_t chain, int32_t *flags);

/* per local chain: mean(-loglik), mean(exp c), mean(exp d) over the samples emitted so far;
 * host arrays of n_chains doubles (any may be NULL).  n_samples receives the divisor. */
int ser_run_chain_stats(ser_run *run, double *e_negloglik, double *e_c, double *e_d, int32_t *n_samples);
/* same E[-logL], written on the run's stream into DEVICE memory (e.g. an NCCL send buffer) */
int ser_run_chain_stats_device(ser_run *run, double *d_e_negloglik);
/* thinned samples of one local chain (needs SER_STORE_FULL; pi alone needs SER_STORE_PI).
 * a,b: [n][M]; pi: [n][N]; c,d,loglik: [n].  Returns the number of samples in *n. */
int ser_run_fetch_samples(ser_run *run, int32_t chain, int32_t *a, int32_t *b, int32_t *pi, double *c,
                          double *d, double *loglik, int32_t *n);
/* manycd = 1 runs (mcmc.c:777-785, :807-815): per-taxon c, d of one chain, M doubles each, file
 * order; ser_run_get_state's cdl then carries taxon 0's c, d -- what compute_exp_data (mcmc.c:56-57)
 * and mcmc_save_chain (mcmc.c:88-89) read.  The fetch returns the per-taxon values of every stored
 * sample, [n][M] each (SER_STORE_FULL), the rows mcmc_save_chain prints for chain_data.csv. */
int ser_run_get_cd(ser_run *run, int32_t chain, double *c, double *d);
int ser_run_fetch_cd_samples(ser_run *run, int32_t chain, double *c, double *d, int32_t *n);

/* ---------------------------------------------------------------- cross-chain steps */
/* choose_chains: population sigma over all n values, keep min-sigma < x < min+sigma, the k
 * smallest, ids ascending.  Host arrays. */
int ser_select_chains(const double *e_negloglik, int32_t n, int32_t k, int32_t *chosen, int32_t *n_chosen,
                      double *min_out, double *sigma_out);
/* same on the device (d_e: n doubles in device memory; d_chosen: k ints, -1 padded; d_info:
 * 3 doubles = n_chosen, min, sigma).  `stream` is a cudaStream_t or NULL. */
int ser_select_chains_device(const double *d_e, int32_t n, int32_t k, int32_t *d_chosen, double *d_info,
                             int32_t device, void *stream);
/* pair-order counts over the stored samples of the chosen chains that live on this run:
 * cnt[c][i][j] = #{samples t : pi_t(i) < pi_t(j)}, diagonal = -T; chosen holds GLOBAL chain ids,
 * entries owned by other ranks (or -1) leave their slab untouched.  d_counts: [k][N][N] int32
 * in DEVICE memory (zero it first; all-reduce it across ranks afterwards). */
int ser_run_po_counts_device(ser_run *run, const int32_t *d_chosen, int32_t k, int32_t *d_counts);
/* host convenience wrapper: chosen / counts in host memory; only the slabs of held chains are written */
int ser_run_po_counts(ser_run *run, const int32_t *chosen, int32_t k, int32_t *counts);
/* script.py:155-175 finalisation incl. the reference's carry-over between chains when faithful != 0 */
int ser_po_finalize(const int32_t *counts, int32_t k, int32_t N, int32_t chains_selected, int32_t faithful,
                    double *po);

/* per-chain sums over the stored thinned samples of the chosen chains owned by this run
 * (GLOBAL ids; others / -1 leave their slab untouched, a held chain's slab is written in full, corr_num included; host memory):
 *   corr_num[c]  = sum_t sum_i i * pi_t(i)   -> mean Pearson r of pi with 0..N-1 (script.py:129-152):
 *                  r = (corr_num/(T*N) - ((N-1)/2)^2) / ((N^2-1)/12), exact because pi_t is a permutation
 *   pi_sum[c][i] = sum_t pi_t(i)   (script.py:230-252)      needs SER_STORE_PI
 *   a_sum[c][m]  = sum_t a_t(m), b_sum likewise (script.py:255-276)   need SER_STORE_FULL; may be NULL
 * n_samples receives T. */
int ser_run_posterior_sums(ser_run *run, const int32_t *chosen, int32_t k, int64_t *corr_num, int32_t *pi_sum,
                           int32_t *a_sum, int32_t *b_sum, int32_t *n_samples);

/* Convergence diagnostics over the stored samples (DESIGN.md section 3.7).  Quantity q of sample t:
 *   q = 0 -loglik, q = 1 exp(c), q = 2 exp(d) (a manycd run: taxon 0's c, d, as in the exp_data sums); q = 3 + i pi_t(i) */
#define SER_DIAG_SCALARS 1 /* q = 0..2: -loglik, exp(c), exp(d)   (needs SER_STORE_FULL) */
#define SER_DIAG_SITES 2   /* q = 3+i: pi(i)                       (needs SER_STORE_PI)   */
/* per chosen chain (GLOBAL ids; -1 / not held: slab untouched) and quantity, over its T stored samples:
 * stats [k][3+N][4] = mean, var, ess, lags;  halves [k][3+N][4] = mean1, var1, mean2, var2;  n_samples [k] = T.
 * var has divisor T-1; the halves are the first and last floor(T/2) samples (divisor n-1).  ess is Geyer's initial monotone
 * sequence estimate of one chain (no rank normalisation) over lags below min(T, max_lag) (max_lag 0 = no cap); lags = the number
 * of autocorrelations summed -- when it reaches 2 floor(L/2) the cap cut the sequence and ess is an upper bound.  A quantity
 * constant in a chain has var 0, ess NaN, lags 0.  Host memory; quantities `what` does not request keep their slab.
 * SER_E_ARG: k < 1, what not in 1..3, max_lag < 0.  SER_E_STATE: a store below what `what` needs, an accumulating run, a run
 * not initialised, or a chosen chain this run holds with T < 4 (the outputs are then left as they were). */
int ser_run_diagnostics(ser_run *run, const int32_t *chosen, int32_t k, int32_t what, int32_t max_lag, double *stats, double *halves,
                        int32_t *n_samples);
/* split-R-hat per quantity from the halves of k chains (BDA3 section 11.4; host only, no CUDA call): W = mean of the 2k half
 * variances, B/n = variance of the 2k half means (divisor 2k-1), R-hat = sqrt(((n-1)/n W + B/n) / W); NaN where W = 0.
 * SER_E_ARG when the chains' T differ or T < 4. */
int ser_split_rhat(const double *halves, const int32_t *n_samples, int32_t k, int32_t Q, double *rhat);

/* alive[c][j][m] = #{t : a_t(m) <= j <= b_t(m)} over the stored samples of the chosen chains owned by
 * this run (same slab convention as above; int32 [k][N][M], host memory; needs SER_STORE_FULL).
 * The counts behind plot_taxa_occurence_probability_matrix, plot_false_taxa_occurence_probability
 * and plot_false_ones_probability (script.py:306-448): alive, T - alive, X * (T - alive). */
int ser_run_alive_counts(ser_run *run, const int32_t *chosen, int32_t k, int32_t *alive, int32_t *n_samples);

/* Posterior marginals (DESIGN.md section 3.8).  For chosen chain c over its T samples t (T = that chain's own count):
 *   pos[c][i][p]    = #{t : pi_t(i) = p}   site i in file order, position p in [0, N); every row sums to T    (needs SER_STORE_PI)
 *   a_hist[c][m][j] = #{t : a_t(m) = j}    taxon m in file order, j in [0, N] (N + 1 bins); b_hist likewise (need SER_STORE_FULL)
 * a and b are the sampler's half-open range: taxon m is alive at positions a <= pos < b.  Exact integer identities:
 *   sum_p p * pos[c][i][p] == pi_sum[c][i] and sum_j j * a_hist[c][m][j] == a_sum[c][m] (b alike) of ser_run_posterior_sums.
 * Counts add over windows, chains and devices.  Chosen ids are GLOBAL; -1 or a chain this run does not hold leaves its slabs untouched
 * and n_samples[c] = 0; a held chain's slabs are written in full.  Host memory: pos [k][N][N], a_hist / b_hist [k][M][N+1] int32, any
 * of the three may be NULL.  On an accumulating run (SER_ACC_POS / SER_ACC_RANGE) T counts every sample taken since accumulation began.
 * Checked before any CUDA call: SER_E_ARG for k < 1, a NULL chosen or n_samples, or all three outputs NULL; SER_E_STATE for a store
 * below what a requested output needs, an accumulating run without the flag of a requested output, or a run not initialised. */
int ser_run_marginals(ser_run *run, const int32_t *chosen, int32_t k, int32_t *pos, int32_t *a_hist, int32_t *b_hist,
                      int32_t *n_samples);
/* Quantiles of histograms (host only, no CUDA call): out[r][q] = the smallest bin b with sum_{j <= b} hist[r][j] >= probs[q] * total_r
 * (the inverse of the empirical CDF, numpy's "inverted_cdf"), -1 for a row whose total is 0.  hist [rows][bins], out [rows][n_probs].
 * SER_E_ARG: rows < 1, bins < 1, n_probs < 1, a NULL pointer, or a probability outside (0, 1] (NaN included). */
int ser_hist_quantiles(const int32_t *hist, int32_t rows, int32_t bins, const double *probs, int32_t n_probs, int32_t *out);

/* CORR_MN (Docs/Report.pdf Table 1; SURVEY section 8f #3): Pearson correlation of the posterior mean
 * position E[pi(site)] over the stored samples of the chosen chains owned by this run with the MN age
 * of the site read from the .sites file (ser_dataset_read_names): the mean over the stored samples of
 * pearsonr(pi_t, x) -- compute_exp_ages (script.py:129-152) with the real chronology in place of the file
 * order -- averaged over the chosen chains this run owns.  sum_t pi_t is reduced on the device (the
 * posterior kernel); every site needs an age.  corr_age: x = -age_ma ("older = earlier position" is
 * positive, like the report), corr_mn: x = the integer MN unit.  Host doubles; needs SER_STORE_PI. */
int ser_run_site_age_corr(ser_run *run, const ser_dataset *ds, const int32_t *chosen, int32_t k, double *corr_age,
                          double *corr_mn, int32_t *n_sites_used);

/* ---------------------------------------------------------------- streaming summaries
 * Flags of ser_run_accumulate and the parts of the one int32 device record per local chain they allocate, in this order: */
#define SER_ACC_PO 1    /* pair-order counts            [N][N]                                            */
#define SER_ACC_SUMS 2  /* pi_sum [N] (corr_num is derived from it on the way out)                          */
#define SER_ACC_AB 4    /* pi_sum [N], then a_sum, b_sum [M] each   (needs SER_STORE_FULL)                  */
#define SER_ACC_ALIVE 8 /* alive difference slab        [N][M]      (needs SER_STORE_FULL)                  */
#define SER_ACC_POS 16  /* position histograms          [N][N]      (ser_run_marginals' pos)                */
#define SER_ACC_RANGE 32 /* a and b histograms          [2][M][N+1] (needs SER_STORE_FULL)                  */
/* From this call on the sample store is a window of cfg->max_samples rows per chain: ser_run_advance / _advance_both split
 * their sampling calls into sweep launches of at most max_samples calls and, after each, add the window's rows of every
 * local chain into the accumulators on the run's stream (no host synchronisation).  ser_run_po_counts(_device),
 * ser_run_posterior_sums, ser_run_alive_counts, ser_run_marginals and ser_run_site_age_corr then return totals over EVERY sample taken since
 * (T = the chain's sample count), with the usual global ids and slab convention; ser_run_fetch_samples /
 * ser_run_fetch_cd_samples return SER_E_STATE (the window is transient), and so does ser_run_cross_chain_async.
 * Call it before the first sampling call (ser_run_init zeroes the accumulators).  Errors: SER_E_STATE on a run that has
 * already sampled, on a store below what the flags need, or a second time; SER_E_ARG for max_samples < 1; SER_E_CUDA with
 * the byte count when an accumulator does not fit (per chain at 2048 x 8192: the alive slab is 64 MB, the a / b histograms 134 MB). */
int ser_run_accumulate(ser_run *run, int32_t what);

/* ---------------------------------------------------------------- cross-chain step, one call
 * E[-logL] of every chain -> (all-gather) -> choose_chains(k) -> pair-order counts of the chosen chains
 * -> (all-reduce), enqueued back to back on the run's stream: no host synchronisation between the
 * kernels and the collectives.  comm == NULL: this run holds all the chains.  With a communicator the
 * chains of rank r are the global ids [r * n_chains, (r+1) * n_chains) (every rank the same n_chains).
 * ser_run_cross_chain_async only enqueues; ser_run_cross_chain_result waits and copies to the host:
 * chosen[k] (GLOBAL ids, ascending, -1 padded), counts [k][N][N] (may be NULL).
 * Replaces script.py:70-99 + :155-189 over the chains of run_all_chains (:48-67). */
typedef struct ser_comm ser_comm;
int ser_run_cross_chain_async(ser_run *run, ser_comm *comm, int32_t k);
int ser_run_cross_chain_result(ser_run *run, int32_t *chosen, int32_t *n_chosen, double *min_out, double *sigma_out,
                               int32_t *counts);
/* device-side results of the last ser_run_cross_chain_async (valid until the next one / destroy):
 * d_e_all [n_total] doubles, d_chosen [k] ints, d_info [3] doubles, d_counts [k][N][N] ints */
int ser_run_cross_chain_buffers(ser_run *run, double **d_e_all, int32_t **d_chosen, double **d_info, int32_t **d_counts);

/* ---------------------------------------------------------------- multi-GPU, one process per GPU
 * NCCL communicator owned by the library (libnccl.so.2 is loaded on first use).  Rank 0 makes the
 * id, the launcher (torchrun / MPI / a file) broadcasts its SER_COMM_ID_BYTES bytes, every rank
 * calls ser_comm_create.  The collectives of ser_run_cross_chain_async run on the run's stream. */
#define SER_COMM_ID_BYTES 128
int ser_comm_unique_id(uint8_t id[SER_COMM_ID_BYTES]);
int ser_comm_create(const uint8_t id[SER_COMM_ID_BYTES], int32_t n_ranks, int32_t rank, int32_t device, ser_comm **out);
int ser_comm_info(const ser_comm *comm, int32_t *n_ranks, int32_t *rank);
void ser_comm_destroy(ser_comm *comm);

/* ---------------------------------------------------------------- multi-GPU, one process for the box
 * run_all_chains' Pool (script.py:48-67) as ONE call over n_gpus devices: cfg->n_chains is the TOTAL,
 * chains are sharded in contiguous blocks by global id (cfg->chain_offset = id of the first), one host
 * thread drives all devices asynchronously.  The cross-chain step needs no collective library when the
 * devices have peer access (NVLink / NVSwitch): ser_stats kernels store their E[-logL] slice straight
 * into every peer's gather buffer, every device runs the same selection, and the owner of a chosen
 * chain stores its pair-order slab straight into every peer's count buffer; cross-device ordering by
 * CUDA events only.  Without peer access (or SER_MULTI_NCCL=1) the same step runs over
 * ncclCommInitAll communicators.  devices == NULL: 0 .. n_gpus-1. */
typedef struct ser_multi ser_multi;
int ser_multi_create(const ser_dataset *ds, const ser_run_config *cfg, int32_t n_gpus, const int32_t *devices, ser_multi **out);
void ser_multi_destroy(ser_multi *m);
int ser_multi_init(ser_multi *m);
int ser_multi_advance(ser_multi *m, int32_t burn_calls, int32_t sample_calls);
int ser_multi_sync(ser_multi *m);
/* max over the devices of the CUDA-event time of the kernels launched since creation / last reset */
int ser_multi_elapsed_ms(ser_multi *m, double *ms, int32_t reset);
int ser_multi_layout(const ser_multi *m, int32_t *n_gpus, int32_t *chains_per_gpu, int32_t *uses_peer_stores);
/* the run that owns a GLOBAL chain id, and the chain's local index there (for ser_run_get_state, the writers, ...) */
int ser_multi_locate(ser_multi *m, int32_t global_chain, ser_run **run, int32_t *local_chain);
int ser_multi_check(ser_multi *m, int32_t *n_bad);
/* per chain (global order): mean(-loglik), mean(exp c), mean(exp d); host arrays of n_chains doubles (may be NULL) */
int ser_multi_chain_stats(ser_multi *m, double *e_negloglik, double *e_c, double *e_d, int32_t *n_samples);
/* the whole cross-chain step; results as ser_run_cross_chain_result */
int ser_multi_cross_chain(ser_multi *m, int32_t k, int32_t *chosen, int32_t *n_chosen, double *min_out, double *sigma_out,
                          int32_t *counts);

/* ---------------------------------------------------------------- checkpoints
 * Every chain of a run written to one file and read back into another run, in another process, on any number of devices:
 * the chains continue bit for bit.  The file is keyed by global chain id, so a file saved from a ser_multi over 8 GPUs
 * loads into a ser_multi over 1, 2 or 4, into a ser_run, or into a subset run (ser_run_create_chains), each reading only the
 * records of its own chains.  Format, size and what is validated: DESIGN.md section 3.6.
 *
 * Save waits for the run's stream, writes path.tmp, syncs it to disk and renames it over path (a crash mid-write keeps the
 * previous file).  The same chains in the same state give a byte-identical file whatever the sharding or the sweep path.
 *
 * Load stands in for the init call on a created run, fresh or initialised.  In replay mode set the tapes first; a run that
 * is to accumulate calls ser_run_accumulate first with the flags it was saved with.  On any error the run is left
 * uninitialised (advance returns SER_E_STATE); nothing is swept on a state that failed a check:
 *   SER_E_IO     missing or truncated file, bad magic or version, checksum mismatch
 *   SER_E_ARG    another dataset (fingerprint of X and the hard flags, or N / M), or a local chain's global id not in the file
 *   SER_E_STATE  mode, seed, sweeps_per_call, manycd, store, max_samples or accumulate flags differ from the run's
 *   SER_E_TAPE   a replay cursor beyond the chain's tape
 *   SER_E_CHECK  a record out of range (a <= b <= N, rpi a permutation; the same for each stored sample row the chain holds)
 *                or failing the consistency check (ser_run_check's)
 * One process per GPU: each rank saves and loads its own file with the ser_run_* pair. */
int ser_run_save_checkpoint(ser_run *run, const char *path);
int ser_run_load_checkpoint(ser_run *run, const char *path);
int ser_multi_save_checkpoint(ser_multi *m, const char *path);
int ser_multi_load_checkpoint(ser_multi *m, const char *path);
/* header only, host only, no CUDA call: what a resume needs to plan the remaining calls.  calls_done counts the calls
 * advanced since init (burn-in and sampling), n_samples the sampling calls.  Any pointer may be NULL. */
int ser_checkpoint_info(const char *path, int32_t *N, int32_t *M, int32_t *n_chains, int64_t *calls_done,
                        int32_t *n_samples, uint32_t *seed, int32_t *mode, int32_t *manycd);

/* ---------------------------------------------------------------- reference-compatible files */
/* Writes Chains-style files for one local chain into `dir` (which must exist, like the
 * reference): chain_data.csv, exp_data.csv, taxa.csv, sites.csv, hard_sites.csv. */
int ser_write_chain_files(ser_run *run, int32_t chain, const char *dir);

/* Labelled companions of taxa.csv / sites.csv for a dataset that carries names
 * (ser_dataset_read_names): taxa_named.csv "taxon,a,b" and sites_named.csv
 * "site,mn_unit,age_ma,hard,pi" (final state of one local chain). */
int ser_write_labelled_files(ser_run *run, int32_t chain, const ser_dataset *ds, const char *dir);

/* micro-benchmarks of the SM-local ceilings the sweep is bound by (DESIGN.md "roofline"):
 * out[0] = fp64 FMA TFLOP/s, out[1] = shared-memory load GB/s, out[2] = popc Gop/s */
int ser_microbench(int32_t device, double out[3]);
/* the same plus out[3..5] = the kernel times (ms) behind the three rates, so the peaks can be re-derived:
 * work = 2 x SMs x 1024 threads x 20 000 iterations x {8 FMA = 16 flop, (1/4 of the iterations) 8 x 16 B, 8 popc} */
int ser_microbench_ex(int32_t device, double out[6]);

#ifdef __cplusplus
}
#endif
#endif /* SERIATION_B200_H */
