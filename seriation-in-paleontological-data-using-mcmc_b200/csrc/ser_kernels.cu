/*
 * ser_kernels.cu -- sm_100a kernels of the seriation sweep and the run object behind the C ABI.
 *
 * Mapping: one CTA per chain, one thread per taxon (+ one thread owning the hard-site mask).
 * The chain's occurrence matrix lives in shared memory as position-ordered bit columns
 * V[word][column]; a/b of a taxon live in its thread's registers.  A sweep is
 *   stage draws -> c,d -> a/b Gibbs (per thread) -> 16 pi proposals (per-thread integer deltas,
 *   REDUX + one __syncthreads, redundant uniform decision, per-thread column update on accept).
 * No tensor cores, no global traffic inside a sweep except the draw tape (replay) and the
 * thinned samples.  See DESIGN.md for the layout and the roofline that bounds each phase.
 *
 * Reference: /root/reference/C_Implementation/mcmc.c (line numbers next to each device function).
 */
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cfloat>
#include <climits>
#include <cstring>
#include <vector>

#include "ser_chain_core.h"
#include "ser_internal.h"

#define SER_MINC (-6.9077552789821368)
#define SER_MAXC (-2.3025850929940455)
#define SER_MIND (-1.6094379124341003)
#define SER_MAXD (-0.22314355131420971)

#define SER_PI_DRAWS 72 /* >= 4 + 5*13 = 69 draws a sweep's pi part can consume */
#define SER_MAX_WARPS 32
#define SER_MAX_GROUPS 8 /* column groups the item weights of a Gibbs step are evaluated in */

#include "ser_device_common.cuh"
#include "ser_sweep_kernel.cuh"
#include "ser_sweep_kernel_big.cuh"
#include "ser_aux_kernels.cuh"

/* ================================================================== host side: the run object */
/* The sweep kernel instantiations a run can launch.  One thread per taxon, [manycd][variant]: variant 0 = 64 registers, any
 * block size; variant 1 = 80 registers, blocks of <= 384 threads, two of them resident.  Large shapes, [warp][manycd]: the Gibbs
 * phase in CTA-wide column groups (warp = 0) or in warp batches (1).  The entries' order is the order the instantiations are
 * compiled in, and it matters: with <false, true> listed before <true, false>, those two get another register allocation. */
typedef void (*SweepFn)(KParams);
static const SweepFn SWEEP_SMALL[2][2] = {{ser_sweep_kernel<1024, 1, false>, ser_sweep_kernel<384, 2, false>},
                                          {ser_sweep_kernel<1024, 1, true>, ser_sweep_kernel<384, 2, true>}};
static const SweepFn SWEEP_BIG[2][2] = {{ser_sweep_kernel_big<false, false>, ser_sweep_kernel_big<true, false>},
                                        {ser_sweep_kernel_big<false, true>, ser_sweep_kernel_big<true, true>}};

#define CUDA_TRY(expr)                                                                          \
  do {                                                                                          \
    cudaError_t e__ = (expr);                                                                   \
    if (e__ != cudaSuccess) {                                                                   \
      ser_set_error("CUDA error %s at %s:%d: %s", cudaGetErrorName(e__), __FILE__, __LINE__, cudaGetErrorString(e__)); \
      return SER_E_CUDA;                                                                        \
    }                                                                                           \
  } while (0)

struct ser_run {
  ser_run_config cfg;
  KParams kp;
  int N, M, W, C, nh;
  uint8_t *h_hard;
  uint32_t *d_Xs;
  uint8_t *d_hard;
  int *d_ones, *d_off;
  uint16_t *d_order;
  uint32_t *d_item_col;
  uint2 *d_unit_tab;
  uint32_t *d_hbits;
  uint16_t *d_col_sites;
  uint16_t *d_ab, *d_rpi;
  ChainScalars *d_scal;
  double *d_tape;
  unsigned long long *d_tape_off;
  uint16_t *d_samp_a, *d_samp_b, *d_samp_pi;
  double *d_samp_cdl, *d_cd4, *d_samp_cd_all;
  int *d_scratch_i; /* export buffers: a,b,pi,rpi,cnt[4M] */
  int *d_bad;
  cudaStream_t stream;
  cudaEvent_t ev_start, ev_stop;
  int timing_open;
  double elapsed_ms;
  long long launches;
  size_t smem_init, smem_small;
  int Caux, big, big_threads;
  uint32_t *d_gV;
  uint16_t *d_gpre;
  int *d_bgrp;
  int4 *d_bbat;
  int big_warp; /* the Gibbs phase of the large-shape kernel runs warp batches (else CTA-wide column groups) */
  /* the sweep kernel instantiation the run launches (SWEEP_SMALL / SWEEP_BIG), its block size and dynamic shared memory */
  SweepFn sweep_fn;
  int sweep_block;
  size_t sweep_smem;
  int sweep_slots; /* resident CTAs of sweep_fn on the whole device; on the large-shape path no more than chains (one gV slot each) */
  int initialized, have_tapes;
  /* persistent work-queue grid of ser_sweep_kernel: (chain, chunk of calls) items, see ser_run_advance_both */
  uint32_t *d_V;            /* [chain][W][C] bit columns carried between work items */
  unsigned int *d_queue;    /* next work item of the running launch */
  unsigned int *d_done;     /* [chain] work items completed since init (monotonic) */
  unsigned int chunks_done; /* host mirror: items every chain has completed before the next launch */
  /* cross-chain step on the run's stream (ser_run_cross_chain_async) */
  double *d_e_all, *d_info;
  int *d_chosen, *d_counts;
  int cc_k, cc_total, cc_ranks, cc_rank, cc_valid;
  /* CUDA-event pairs around every sweep launch since the last reset (ser_run_sweep_time): read after the fact, so
   * timing the dominant kernel does not put a host synchronisation into the timed region */
  std::vector<cudaEvent_t> *sweep_ev;
  size_t sweep_ev_used;
  /* subset runs (ser_run_create_chains): global id of every local chain, device copy in kp.chain_ids */
  int *h_chain_ids, *d_chain_ids;
  /* streaming accumulators (ser_run_accumulate): SER_ACC_* flags, one record per local chain [n][acc_layout().ints] */
  int acc_what, sampled;
  int *d_acc;
  /* checkpoints (ser_ckpt.cuh): calls and sampling calls advanced since init, and the fingerprint of the run's dataset */
  long long calls_done;
  int samples_done;
  uint64_t ds_fp;
};

/* multi-GPU pieces (ser_multi.cuh): NCCL entry points resolved at run time */
struct ser_comm;
static int comm_all_gather_e(ser_comm *comm, double *d_e_all, int n_local, cudaStream_t stream);
static int comm_all_reduce_counts(ser_comm *comm, int *d_counts, size_t n, cudaStream_t stream);
static int comm_ranks(const ser_comm *comm, int *n_ranks, int *rank);
static uint64_t ckpt_dataset_fingerprint(const ser_dataset *ds); /* ser_ckpt.cuh */

/* Stream-ordered pool allocation: cudaMalloc/cudaFree are synchronous driver calls with erratic
 * latency (tens to hundreds of ms on shared hosts).  The library allocates from its OWN memory pool per
 * device (not the process-wide default pool other allocators share), with a bounded release threshold:
 * up to SER_POOL_KEEP_MB (default 1024) of freed blocks stay cached, so creating / destroying runs and
 * the temporary buffers of the cross-chain steps cost microseconds after the first use, while a
 * multi-GB sample store goes back to the driver when its run is destroyed. */
#include <mutex>
static cudaError_t pool_alloc(void **ptr, size_t bytes, cudaStream_t stream)
{
  static std::mutex mu;
  static cudaMemPool_t pools[64] = {nullptr};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  cudaMemPool_t pool = nullptr;
  if (dev >= 0 && dev < 64) {
    std::lock_guard<std::mutex> lock(mu);
    if (!pools[dev]) {
      cudaMemPoolProps props;
      memset(&props, 0, sizeof(props));
      props.allocType = cudaMemAllocationTypePinned;
      props.handleTypes = cudaMemHandleTypeNone;
      props.location.type = cudaMemLocationTypeDevice;
      props.location.id = dev;
      if (cudaMemPoolCreate(&pools[dev], &props) == cudaSuccess) {
        unsigned long long keep = 1024ull << 20;
        if (const char *v = getenv("SER_POOL_KEEP_MB")) keep = (unsigned long long)atoll(v) << 20;
        cudaMemPoolSetAttribute(pools[dev], cudaMemPoolAttrReleaseThreshold, &keep);
      } else {
        pools[dev] = nullptr;
        cudaGetLastError();
      }
    }
    pool = pools[dev];
  }
  if (pool) return cudaMallocFromPoolAsync(ptr, bytes ? bytes : 1, pool, stream);
  return cudaMallocAsync(ptr, bytes ? bytes : 1, stream);
}
#define POOL_ALLOC(ptr, bytes) pool_alloc((void **)(ptr), (bytes), run->stream)

static int set_device(const ser_run *run) { CUDA_TRY(cudaSetDevice(run->cfg.device)); return SER_OK; }

static void mark_launch(ser_run *run)
{
  if (!run->timing_open) { cudaEventRecord(run->ev_start, run->stream); run->timing_open = 1; }
  run->launches++;
}

/* Every kernel with dynamic shared memory may use up to the sm_100 opt-in maximum.  The attribute is a
 * property of the FUNCTION (not of a run): sized per run it would be lowered by the next run of a smaller
 * dataset and make the launches of a live larger one fail, so it is set to the maximum once and the launches
 * pass each run's own size. */
#define SER_SMEM_OPTIN (227 * 1024)
#define SER_SMEM_DYN_MAX (SER_SMEM_OPTIN - 1024) /* the sweep kernels hold 1 KB of static shared memory */
static cudaError_t allow_max_dynamic_smem(void)
{
  /* once per device: driver calls that run creation (the e2e path creates a run per job) need not repeat */
  static std::mutex mu;
  static bool done[64] = {false};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  std::lock_guard<std::mutex> lock(mu);
  if (dev >= 0 && dev < 64 && done[dev]) return cudaSuccess;
  auto allow = [&](const void *f) { /* static + dynamic shared memory share the opt-in limit */
    cudaFuncAttributes fa;
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, f);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, SER_SMEM_OPTIN - (int)fa.sharedSizeBytes);
  };
  allow((const void *)ser_init_kernel);
  for (int m = 0; m < 2; m++)
    for (int v = 0; v < 2; v++) {
      allow((const void *)SWEEP_SMALL[m][v]);
      allow((const void *)SWEEP_BIG[m][v]);
    }
  if (e == cudaSuccess && dev >= 0 && dev < 64) done[dev] = true;
  return e;
}

/* Warp batches of the large-shape kernel's Gibbs phase (ser_sweep_kernel_big<.., WB = true>): off[c] = first item of sorted column c
 * (a column has ones + 1 items), wcap = items a warp's slice of the item buffers holds (>= the widest column).  A batch = consecutive
 * columns whose items fit the slice, at most 32; a column gets 32 / columns lanes, rounded down to a power of two.  When the columns
 * that fit would leave more than 32 - minlanes lanes idle, the batch shrinks to a power of two of columns (all 32 lanes busy).
 * Entry = {first column, columns | lane shift << 16, first item, last item + 1}. */
static void plan_warp_batches(const int *off, int M, long long wcap, int minlanes, std::vector<int4> &out)
{
  out.clear();
  for (int c0 = 0; c0 < M;) {
    int c1 = c0;
    while (c1 < M && c1 - c0 < 32 && off[c1 + 1] - off[c0] <= wcap) c1++;
    int nc = c1 - c0, lsh = 0;
    while ((nc << (lsh + 1)) <= 32) lsh++;
    if ((nc << lsh) < minlanes) {
      int p2 = 1;
      while (p2 * 2 <= nc) p2 *= 2;
      if (c0 + p2 < M) { nc = p2; lsh = 0; while ((nc << (lsh + 1)) <= 32) lsh++; }
    }
    c1 = c0 + nc;
    out.push_back(make_int4(c0, nc | (lsh << 16), off[c0], off[c1]));
    c0 = c1;
  }
}

/* the same plan from the columns' occurrence counts (host only, no device needed): what a run of such a matrix would use */
extern "C" int ser_plan_warp_batches(const int32_t *ones_sorted, int32_t M, int32_t wcap, int32_t *batches, int32_t max_batches, int32_t *n_batches)
{
  if (!ones_sorted || M < 1 || wcap < 1 || !n_batches) { ser_set_error("ser_plan_warp_batches: bad argument"); return SER_E_ARG; }
  std::vector<int> off((size_t)M + 1, 0);
  for (int c = 0; c < M; c++) {
    if (ones_sorted[c] < 0 || ones_sorted[c] + 1 > wcap) { ser_set_error("ser_plan_warp_batches: column %d has %d items, a slice holds %d", c, ones_sorted[c] + 1, wcap); return SER_E_ARG; }
    off[c + 1] = off[c] + ones_sorted[c] + 1;
  }
  std::vector<int4> plan;
  plan_warp_batches(off.data(), M, wcap, 28, plan);
  *n_batches = (int32_t)plan.size();
  if (batches) {
    if ((int)plan.size() > max_batches) { ser_set_error("ser_plan_warp_batches: %zu batches, room for %d", plan.size(), max_batches); return SER_E_ARG; }
    for (size_t b = 0; b < plan.size(); b++) { batches[4 * b] = plan[b].x; batches[4 * b + 1] = plan[b].y; batches[4 * b + 2] = plan[b].z; batches[4 * b + 3] = plan[b].w; }
  }
  return SER_OK;
}

/* Column groups of the Gibbs step: the item weights of a step go through a buffer of Ival doubles,
 * one group of columns at a time.  Fewer, larger groups = fewer barriers; a smaller buffer = more
 * resident chains per SM (measured on B200: +15-20 % per extra resident CTA, -4 % per extra group).
 * Take the fewest groups that reach the best residency; SER_SWEEP_GROUPS forces a count. */
template <typename K>
static int choose_groups(KParams &kp, const std::vector<int> &off, int M, int N, int W, int C, int manycd, K kernel, size_t *smem_out)
{
  int best_occ = 0, force = 0;
  if (const char *v = getenv("SER_SWEEP_GROUPS")) force = std::max(1, std::min(SER_MAX_GROUPS, atoi(v)));
  for (int G = 1; G <= SER_MAX_GROUPS; G++) {
    if (force && G != force) continue;
    int gc[SER_MAX_GROUPS + 1], ge[SER_MAX_GROUPS + 1], ng = 0, ival = 0;
    gc[0] = 0; ge[0] = 0;
    for (int c = 0; c < M && ng < G; c++) /* close a group at the column where its share of the items is reached */
      if (c + 1 == M || off[c + 1] >= (long long)kp.I * (ng + 1) / G) {
        ng++; gc[ng] = c + 1; ge[ng] = off[c + 1];
        ival = std::max(ival, ge[ng] - ge[ng - 1]);
      }
    const size_t sz = smem_layout(nullptr, nullptr, N, W, C, kp.I, manycd, ival);
    if (sz > SER_SMEM_DYN_MAX) continue;
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, C, sz) != cudaSuccess) {
      ser_set_error("ser_run_create: occupancy query failed: %s", cudaGetErrorString(cudaGetLastError()));
      return SER_E_CUDA;
    }
    if (occ > best_occ) {
      best_occ = occ;
      kp.n_groups = ng; kp.Ival = ival;
      memcpy(kp.grp_c, gc, sizeof(gc)); memcpy(kp.grp_e, ge, sizeof(ge));
      *smem_out = sz;
    }
  }
  if (!best_occ) { ser_set_error("ser_run_create: the chain state does not fit shared memory"); return SER_E_ARG; }
  return SER_OK;
}

/* builds `run` in place; on any failure the caller (ser_run_create) releases whatever exists so far */
static int run_create_impl(const ser_dataset *ds, const ser_run_config *cfg, ser_run *run)
{
  const int N = ds->N, M = ds->M;
  run->cfg = *cfg;
  run->N = N; run->M = M; run->nh = ds->nh;
  run->W = N / 32 + 1;
  run->C = ((M + 1) + 31) / 32 * 32;
  run->Caux = std::min(1024, (M + 31) / 32 * 32);
  /* large-shape path when one thread per column does not fit a CTA or its shared memory;
   * SER_FORCE_BIG=<threads> forces it (tests run the whole parity suite through it) */
  run->big_threads = 1024;
  if (const char *fb = getenv("SER_FORCE_BIG")) { run->big = 1; if (atoi(fb) >= 32) run->big_threads = std::min(1024, atoi(fb) / 32 * 32); }
  if (run->C > 1024) { run->big = 1; run->C = 1024; }
  if (const char *bt = getenv("SER_BIG_THREADS")) { if (atoi(bt) >= 32) run->big_threads = std::min(1024, atoi(bt) / 32 * 32); }
  CUDA_TRY(cudaSetDevice(cfg->device));
  CUDA_TRY(cudaStreamCreateWithFlags(&run->stream, cudaStreamNonBlocking));
  CUDA_TRY(cudaEventCreate(&run->ev_start));
  CUDA_TRY(cudaEventCreate(&run->ev_stop));

  KParams &kp = run->kp;
  memset(&kp, 0, sizeof(kp));
  kp.N = N; kp.M = M; kp.W = run->W; kp.C = run->C; kp.nh = ds->nh;
  kp.Mw = (M + 31) / 32; kp.Npad = (N + 7) / 8 * 8; kp.Mpad = (M + 7) / 8 * 8;
  kp.mode = cfg->mode; kp.chain_offset = cfg->chain_offset; kp.seed = cfg->seed;
  kp.sweeps_per_call = cfg->sweeps_per_call; kp.store = cfg->store; kp.max_samples = cfg->max_samples;
  /* initial c, d and the flooring constant with the HOST libm: the bits the reference gets */
  kp.c0 = log(.01); kp.d0 = log(.3);
  kp.cc0 = log(1. - exp(kp.c0)); kp.dd0 = log(1. - exp(kp.d0));
  if (cfg->mode == SER_MODE_FREE) {
    /* free-running chains derive log(1 - e^c) with the bit-reproducible log / exp everywhere, also for the
     * initial values (a d that never moves keeps this companion for the whole run): what the oracle's
     * reproduction of the stream evaluates.  Replay keeps the host libm's bits, i.e. the reference's. */
    kp.cc0 = ser_log(SER_SUB(1.0, ser_exp(kp.c0)));
    kp.dd0 = ser_log(SER_SUB(1.0, ser_exp(kp.d0)));
  }
  kp.eps = exp(-32.236191301916641); /* exp(LOGEPSILON), mcmc.h:26 */

  /* Columns = taxa sorted by number of occurrences (descending), so that the threads of a warp
   * own taxa with similar item counts; `order` maps a column back to its taxon.  Site-major bit
   * matrix over columns, ones per column, and the static item tables of the Gibbs step. */
  std::vector<int> tones(M, 0);
  long long ones_total = 0;
  for (int n = 0; n < N; n++)
    for (int m = 0; m < M; m++)
      if (ds->X[(size_t)n * M + m]) { tones[m]++; ones_total++; }
  std::vector<uint16_t> order(M);
  for (int m = 0; m < M; m++) order[m] = (uint16_t)m;
  std::stable_sort(order.begin(), order.end(), [&](uint16_t x, uint16_t y) { return tones[x] > tones[y]; });
  std::vector<uint32_t> Xs((size_t)N * kp.Mw, 0u);
  std::vector<int> ones(M, 0), off(M + 1, 0);
  for (int c = 0; c < M; c++) {
    ones[c] = tones[order[c]];
    off[c + 1] = off[c] + ones[c] + 1;
    for (int n = 0; n < N; n++)
      if (ds->X[(size_t)n * M + order[c]]) Xs[(size_t)n * kp.Mw + (c >> 5)] |= 1u << (c & 31);
  }
  kp.I = off[M];
  for (int c = 0; c < M; c++) if (order[c] == 0) kp.col0 = c;
  std::vector<uint32_t> hbits(M, 0u); /* ones of a column at the hard sites, by hard rank (= file order of the hard sites) */
  {
    int k = 0;
    for (int n = 0; n < N && k < 32; n++)
      if (ds->hard[n]) {
        for (int c = 0; c < M; c++) if (ds->X[(size_t)n * M + order[c]]) hbits[c] |= 1u << k;
        k++;
      }
  }
  std::vector<uint16_t> col_sites((size_t)std::max<long long>(1, ones_total));
  for (int c = 0, w = 0; c < M; c++)
    for (int n = 0; n < N; n++)
      if (ds->X[(size_t)n * M + order[c]]) col_sites[w++] = (uint16_t)n;
  std::vector<uint32_t> item_col(kp.I);
  for (int c = 0; c < M; c++)
    for (int e = off[c]; e < off[c + 1]; e++) item_col[e] = ((uint32_t)c << 16) | (uint32_t)(e - off[c]);
  kp.ones_total = ones_total;
  run->h_hard = (uint8_t *)malloc(N);
  if (!run->h_hard) { ser_set_error("ser_run_create: out of memory"); return SER_E_ARG; }
  memcpy(run->h_hard, ds->hard, N);
  run->ds_fp = ckpt_dataset_fingerprint(ds);

  const size_t nc = (size_t)cfg->n_chains;
  CUDA_TRY(POOL_ALLOC(&run->d_Xs, Xs.size() * 4));
  CUDA_TRY(POOL_ALLOC(&run->d_hard, N));
  CUDA_TRY(POOL_ALLOC(&run->d_ones, M * sizeof(int)));
  CUDA_TRY(POOL_ALLOC(&run->d_off, (M + 1) * sizeof(int)));
  CUDA_TRY(POOL_ALLOC(&run->d_order, M * sizeof(uint16_t)));
  CUDA_TRY(POOL_ALLOC(&run->d_item_col, (size_t)kp.I * sizeof(uint32_t)));
  CUDA_TRY(POOL_ALLOC(&run->d_col_sites, col_sites.size() * sizeof(uint16_t)));
  CUDA_TRY(cudaMemcpyAsync(run->d_col_sites, col_sites.data(), col_sites.size() * sizeof(uint16_t), cudaMemcpyHostToDevice, run->stream));
  CUDA_TRY(POOL_ALLOC(&run->d_hbits, (size_t)M * sizeof(uint32_t)));
  CUDA_TRY(cudaMemcpyAsync(run->d_hbits, hbits.data(), (size_t)M * sizeof(uint32_t), cudaMemcpyHostToDevice, run->stream));
  CUDA_TRY(POOL_ALLOC(&run->d_ab, nc * 2 * kp.Mpad * sizeof(uint16_t)));
  CUDA_TRY(POOL_ALLOC(&run->d_rpi, nc * kp.Npad * sizeof(uint16_t)));
  CUDA_TRY(POOL_ALLOC(&run->d_scal, nc * sizeof(ChainScalars)));
  CUDA_TRY(POOL_ALLOC(&run->d_scratch_i, (size_t)(2 * N + 6 * M + 16) * sizeof(int)));
  CUDA_TRY(POOL_ALLOC(&run->d_bad, sizeof(int)));
  CUDA_TRY(cudaMemcpyAsync(run->d_Xs, Xs.data(), Xs.size() * 4, cudaMemcpyHostToDevice, run->stream));
  CUDA_TRY(cudaMemcpyAsync(run->d_hard, ds->hard, N, cudaMemcpyHostToDevice, run->stream));
  CUDA_TRY(cudaMemcpyAsync(run->d_ones, ones.data(), M * sizeof(int), cudaMemcpyHostToDevice, run->stream));
  CUDA_TRY(cudaMemcpyAsync(run->d_off, off.data(), (M + 1) * sizeof(int), cudaMemcpyHostToDevice, run->stream));
  CUDA_TRY(cudaMemcpyAsync(run->d_order, order.data(), M * sizeof(uint16_t), cudaMemcpyHostToDevice, run->stream));
  CUDA_TRY(cudaMemcpyAsync(run->d_item_col, item_col.data(), (size_t)kp.I * sizeof(uint32_t), cudaMemcpyHostToDevice, run->stream));
  CUDA_TRY(cudaMemsetAsync(run->d_scal, 0, nc * sizeof(ChainScalars), run->stream));
  CUDA_TRY(cudaStreamSynchronize(run->stream));
  if (cfg->store >= SER_STORE_PI && cfg->max_samples > 0) {
    CUDA_TRY(POOL_ALLOC(&run->d_samp_pi, nc * cfg->max_samples * N * sizeof(uint16_t)));
  }
  if (cfg->store >= SER_STORE_FULL && cfg->max_samples > 0) {
    CUDA_TRY(POOL_ALLOC(&run->d_samp_a, nc * cfg->max_samples * M * sizeof(uint16_t)));
    CUDA_TRY(POOL_ALLOC(&run->d_samp_b, nc * cfg->max_samples * M * sizeof(uint16_t)));
    CUDA_TRY(POOL_ALLOC(&run->d_samp_cdl, nc * cfg->max_samples * 3 * sizeof(double)));
  }
  kp.Xs = run->d_Xs; kp.hard = run->d_hard; kp.ones = run->d_ones;
  kp.order = run->d_order; kp.off = run->d_off; kp.item_col = run->d_item_col; kp.hbits = run->d_hbits; kp.col_sites = run->d_col_sites;
  kp.ab = run->d_ab; kp.rpi = run->d_rpi; kp.scal = run->d_scal;
  kp.samp_a = run->d_samp_a; kp.samp_b = run->d_samp_b; kp.samp_pi = run->d_samp_pi; kp.samp_cdl = run->d_samp_cdl;
  if (cfg->manycd) { /* per-taxon c, d: state rows and, with the full store, per-sample rows */
    kp.manycd = 1;
    CUDA_TRY(POOL_ALLOC(&run->d_cd4, nc * 4 * kp.Mpad * sizeof(double)));
    if (cfg->store >= SER_STORE_FULL && cfg->max_samples > 0)
      CUDA_TRY(POOL_ALLOC(&run->d_samp_cd_all, nc * cfg->max_samples * 2 * M * sizeof(double)));
    kp.cd4 = run->d_cd4; kp.samp_cd_all = run->d_samp_cd_all;
  }

  run->smem_small = aux_layout(nullptr, nullptr, N);
  run->smem_init = run->smem_small + sizeof(double) * 2 * N + sizeof(uint16_t) * 3 * N + 64;
  CUDA_TRY(allow_max_dynamic_smem());
  const int manycd = cfg->manycd;
  if (!run->big) {
    /* one thread per column while the columns, postings and one group's item weights fit shared memory, else (or with
     * SER_FORCE_BIG) the large-shape kernel.  The groups are sized on the 80-register variant for per-taxon c, d in blocks of
     * up to 384 threads, which needs those registers (2.7 M vs 2.5 M sweeps/s on g2s2 with 64), else on the 64-register one.
     * Then the variant with more resident CTAs runs, the roomier one on a tie; SER_SWEEP_VARIANT forces it. */
    const bool fits85 = run->C <= 384;
    const int rc = choose_groups(kp, off, M, N, run->W, run->C, manycd, SWEEP_SMALL[manycd][manycd && fits85], &run->sweep_smem);
    if (rc == SER_E_CUDA) return rc;
    if (rc != SER_OK) run->big = 1;
    else {
      int occ64 = 0, occ85 = 0;
      CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ64, SWEEP_SMALL[manycd][0], run->C, run->sweep_smem));
      if (fits85) CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ85, SWEEP_SMALL[manycd][1], run->C, run->sweep_smem));
      int variant = (occ85 >= occ64 && occ85 > 0) ? 1 : 0;
      if (const char *v = getenv("SER_SWEEP_VARIANT")) variant = (atoi(v) == 1 && fits85) ? 1 : 0;
      run->sweep_fn = SWEEP_SMALL[manycd][variant];
      run->sweep_block = run->C;
    }
  }
  if (run->big) {
    /* column groups of the Gibbs phase: as many items as the shared-memory budget holds
     * (SER_BIG_SMEM_KB, default 220), at most 1024 columns, never splitting a column */
    int budget_kb = 220;
    if (const char *v = getenv("SER_BIG_SMEM_KB")) budget_kb = std::max(16, std::min(224, atoi(v)));
    /* gcap = columns per group (sizes the per-column tables of a group), icap = items per group (val 8 + pos 2 bytes each):
     * start from 512 columns, build the groups, shrink gcap to what the widest group uses and give the bytes to icap */
    int gcap = std::min((M + 31) / 32 * 32, 512);
    long long icap = 0;
    std::vector<int> bgrp;
    for (int pass = 0; pass < 4; pass++) {
      const size_t fixed = big_layout(nullptr, nullptr, N, M, 0, gcap, cfg->manycd, gcap);
      icap = ((long long)budget_kb * 1024 - (long long)fixed - 64) / 10 / 32 * 32;
      icap = std::min<long long>(icap, (long long)(kp.I + 31) / 32 * 32);
      if (icap < std::max(N + 1, M)) { /* one whole column, and the M per-taxon terms of the exact sums */
        ser_set_error("ser_run_create: shape needs %zu B of shared memory per chain before any item", fixed);
        return SER_E_ARG;
      }
      bgrp.clear();
      int widest = 0;
      for (int c0 = 0; c0 < M;) {
        int c1 = c0;
        while (c1 < M && c1 - c0 < gcap && off[c1 + 1] - off[c0] <= icap) c1++;
        bgrp.push_back(c0); bgrp.push_back(off[c0]);
        widest = std::max(widest, c1 - c0);
        c0 = c1;
      }
      bgrp.push_back(M); bgrp.push_back(off[M]);
      const int tight = std::min(gcap, (widest + widest / 8 + 31) / 32 * 32); /* head room: larger groups follow from the larger icap */
      if (tight == gcap) break;
      gcap = tight;
    }
    /* Warp batches (default whenever every column's items fit a warp's slice of the item buffers; SER_BIG_WARP=0 keeps the
     * CTA-wide groups): the item buffers are cut into one slice per warp, the batches come from plan_warp_batches. */
    run->big_warp = 0;
    std::vector<int4> bbat;
    {
      const char *bw = getenv("SER_BIG_WARP");
      const int nwarps = run->big_threads / 32, wgcap = 32 * nwarps;
      const size_t wfixed = big_layout(nullptr, nullptr, N, M, 0, 0, cfg->manycd, wgcap);
      int widest_col = 0, minlanes = 28;
      if (const char *v = getenv("SER_BIG_MINLANES")) minlanes = atoi(v);
      for (int c = 0; c < M; c++) widest_col = std::max(widest_col, off[c + 1] - off[c]);
      long long wcap = ((long long)budget_kb * 1024 - (long long)wfixed - 64) / 10 / nwarps / 8 * 8;
      wcap = std::min<long long>(wcap, (long long)(kp.I + 7) / 8 * 8);
      /* val also holds the M per-taxon terms of the exact sums */
      const long long wicap = std::max<long long>(wcap * nwarps, (std::max(N + 1, M) + 31) / 32 * 32);
      if (!(bw && atoi(bw) == 0) && wcap >= widest_col &&
          big_layout(nullptr, nullptr, N, M, (int)wicap, 0, cfg->manycd, wgcap) <= (size_t)budget_kb * 1024) {
        plan_warp_batches(off.data(), M, wcap, minlanes, bbat);
        run->big_warp = 1;
        gcap = 0;
        icap = wicap;
        kp.big_wcap = (int)wcap; kp.big_nb = (int)bbat.size();
        CUDA_TRY(POOL_ALLOC(&run->d_bbat, bbat.size() * sizeof(int4)));
        CUDA_TRY(cudaMemcpyAsync(run->d_bbat, bbat.data(), bbat.size() * sizeof(int4), cudaMemcpyHostToDevice, run->stream));
        kp.bbat = run->d_bbat;
      }
    }
    kp.big_ng = (int)bgrp.size() / 2 - 1; kp.big_icap = (int)icap; kp.big_gcap = gcap;
    CUDA_TRY(POOL_ALLOC(&run->d_bgrp, bgrp.size() * sizeof(int)));
    CUDA_TRY(cudaMemcpyAsync(run->d_bgrp, bgrp.data(), bgrp.size() * sizeof(int), cudaMemcpyHostToDevice, run->stream));
    CUDA_TRY(cudaStreamSynchronize(run->stream));
    kp.bgrp = run->d_bgrp;
    run->sweep_smem = big_layout(nullptr, nullptr, N, M, (int)icap, gcap, cfg->manycd, run->big_warp ? 32 * (run->big_threads / 32) : gcap);
    if (run->sweep_smem > SER_SMEM_DYN_MAX) { ser_set_error("ser_run_create: shape needs %zu B of shared memory per chain", run->sweep_smem); return SER_E_ARG; }
    run->sweep_fn = SWEEP_BIG[run->big_warp][manycd];
    run->sweep_block = run->big_threads;
  }
  kp.n_chains = cfg->n_chains;
  int per_sm = 1, n_sm = 1;
  CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, run->sweep_fn, run->sweep_block, run->sweep_smem));
  CUDA_TRY(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, cfg->device));
  run->sweep_slots = std::max(1, per_sm * n_sm);
  if (run->big) { /* one global scratch slot per resident CTA */
    run->sweep_slots = std::min(cfg->n_chains, run->sweep_slots);
    kp.Cs = ((M + 1) + 31) / 32 * 32;
    const size_t sl = (size_t)run->sweep_slots;
    CUDA_TRY(POOL_ALLOC(&run->d_gV, sl * run->W * kp.Cs * sizeof(uint32_t)));
    CUDA_TRY(POOL_ALLOC(&run->d_gpre, sl * ((run->W >> SER_BIG_G) + 1) * kp.Cs * sizeof(uint16_t)));
    kp.gV = run->d_gV; kp.gpre = run->d_gpre;
  } else {
    /* Units of the Gibbs phase: a column with many items is served by 2, 4, .. 32 adjacent lanes.  Columns are sorted by
     * occurrence count and every column group starts its own round at lane 0, so inside a group the lane counts are
     * non-increasing and every lane group is aligned inside its warp.  T = items per lane aimed at, chosen per group:
     * the value that minimises the summed critical path of the group's rounds (a round = C units) -- light groups
     * take few items per lane and still fit one round; SER_UNIT_ITEMS forces it. */
    auto lsh_of = [](int items, int T) { int l = 0; while (l < 5 && ((items + (1 << l) - 1) >> l) > T) l++; return l; };
    int forceT = 0;
    if (const char *v = getenv("SER_UNIT_ITEMS")) forceT = std::max(1, atoi(v));
    std::vector<uint2> units;
    kp.grp_u[0] = 0;
    for (int g = 0; g < kp.n_groups; g++) {
      const int c0 = kp.grp_c[g], c1 = kp.grp_c[g + 1];
      int bestT = 1 << 30;
      long long best_cost = -1;
      for (int T = 1; T <= 1024; T++) {
        long long cost = 0;
        int in_round = 0, mx = 0;
        for (int c = c0; c < c1; c++) {
          const int items = ones[c] + 1, l = lsh_of(items, T), chunk = (items + (1 << l) - 1) >> l;
          for (int q = 0; q < (1 << l); q++) {
            if (in_round == run->C) { cost += mx + 6; in_round = 0; mx = 0; } /* + the fixed cost of a round */
            in_round++; mx = std::max(mx, chunk);
          }
        }
        if (in_round) cost += mx + 6;
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; bestT = T; }
        if (c0 < c1 && T >= ones[c0] + 1) break; /* one lane per column from here on */
      }
      if (forceT) bestT = forceT;
      for (int c = c0; c < c1; c++) {
        const int l = lsh_of(ones[c] + 1, bestT);
        for (int q = 0; q < (1 << l); q++) units.push_back(make_uint2((uint32_t)c | ((uint32_t)q << 16) | ((uint32_t)l << 24), (uint32_t)off[c]));
      }
      kp.grp_u[g + 1] = (int)units.size();
    }
    kp.n_units = (int)units.size();
    CUDA_TRY(POOL_ALLOC(&run->d_unit_tab, units.size() * sizeof(uint2)));
    CUDA_TRY(cudaMemcpyAsync(run->d_unit_tab, units.data(), units.size() * sizeof(uint2), cudaMemcpyHostToDevice, run->stream));
    CUDA_TRY(cudaStreamSynchronize(run->stream));
    kp.unit_tab = run->d_unit_tab;
    /* persistent work-queue grid: bit columns carried between work items, queue head, per-chain progress */
    if (const char *v = getenv("SER_SWEEP_SLOTS")) run->sweep_slots = std::max(1, atoi(v));
    CUDA_TRY(POOL_ALLOC(&run->d_V, nc * (size_t)run->W * run->C * sizeof(uint32_t)));
    CUDA_TRY(POOL_ALLOC(&run->d_queue, sizeof(unsigned int)));
    CUDA_TRY(POOL_ALLOC(&run->d_done, nc * sizeof(unsigned int)));
    kp.gVc = run->d_V; kp.queue = run->d_queue; kp.done = run->d_done;
  }
  return SER_OK;
}

extern "C" int ser_run_create(const ser_dataset *ds, const ser_run_config *cfg, ser_run **out)
{
  if (!ds || !cfg || !out) { ser_set_error("ser_run_create: null argument"); return SER_E_ARG; }
  *out = nullptr;
  if (cfg->struct_size != sizeof(ser_run_config)) {
    ser_set_error("ser_run_create: cfg->struct_size is %u, this library's ser_run_config has %zu bytes (set struct_size = sizeof(ser_run_config); "
                  "the caller was built against another header)", cfg->struct_size, sizeof(ser_run_config));
    return SER_E_ARG;
  }
  const int N = ds->N, M = ds->M;
  if (N < 2 || N > SER_MAX_SITES) { ser_set_error("ser_run_create: N=%d outside [2,%d]", N, SER_MAX_SITES); return SER_E_ARG; }
  if (M < 1 || M > SER_MAX_TAXA) { ser_set_error("ser_run_create: M=%d outside [1,%d]", M, SER_MAX_TAXA); return SER_E_ARG; }
  if (cfg->n_chains < 1 || cfg->sweeps_per_call < 1) { ser_set_error("ser_run_create: n_chains and sweeps_per_call must be >= 1"); return SER_E_ARG; }
  if (cfg->mode != SER_MODE_FREE && cfg->mode != SER_MODE_REPLAY) { ser_set_error("ser_run_create: bad mode"); return SER_E_ARG; }
  if (cfg->manycd != 0 && cfg->manycd != 1) { ser_set_error("ser_run_create: manycd must be 0 or 1"); return SER_E_ARG; }
  if (cfg->store < SER_STORE_NONE || cfg->store > SER_STORE_FULL || cfg->max_samples < 0) { ser_set_error("ser_run_create: bad store / max_samples"); return SER_E_ARG; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    ser_set_error("ser_run_create: no CUDA device (this library has no CPU path)");
    return SER_E_CUDA;
  }
  if (cfg->device < 0 || cfg->device >= ndev) { ser_set_error("ser_run_create: device %d of %d", cfg->device, ndev); return SER_E_ARG; }
  ser_run *run = (ser_run *)calloc(1, sizeof(ser_run));
  if (!run) { ser_set_error("ser_run_create: out of memory"); return SER_E_ARG; }
  const int rc = run_create_impl(ds, cfg, run);
  if (rc != SER_OK) { /* single exit for every failure: release the stream, events and buffers made so far */
    char keep[512];
    snprintf(keep, sizeof(keep), "%s", ser_last_error());
    ser_run_destroy(run);
    cudaGetLastError();
    ser_set_error("%s", keep);
    return rc;
  }
  *out = run;
  return SER_OK;
}

extern "C" int ser_run_create_chains(const ser_dataset *ds, const ser_run_config *cfg, const int32_t *chain_ids, int32_t n, ser_run **out)
{
  if (!ds || !cfg || !chain_ids || !out) { ser_set_error("ser_run_create_chains: null argument"); return SER_E_ARG; }
  *out = nullptr;
  if (n < 1 || n != cfg->n_chains) { ser_set_error("ser_run_create_chains: %d chain ids for cfg->n_chains = %d", n, cfg->n_chains); return SER_E_ARG; }
  if (cfg->chain_offset != 0) { ser_set_error("ser_run_create_chains: cfg->chain_offset is %d; it must be 0 (chain_ids are the global ids)", cfg->chain_offset); return SER_E_ARG; }
  std::vector<int> sorted(chain_ids, chain_ids + n);
  std::sort(sorted.begin(), sorted.end());
  if (sorted[0] < 0) { ser_set_error("ser_run_create_chains: chain id %d is negative", sorted[0]); return SER_E_ARG; }
  for (int c = 1; c < n; c++)
    if (sorted[c] == sorted[c - 1]) { ser_set_error("ser_run_create_chains: chain id %d is listed twice", sorted[c]); return SER_E_ARG; }
  ser_run *run = nullptr;
  int rc = ser_run_create(ds, cfg, &run);
  if (rc != SER_OK) return rc;
  auto attach = [&]() -> int {
    run->h_chain_ids = (int *)malloc((size_t)n * sizeof(int));
    if (!run->h_chain_ids) { ser_set_error("ser_run_create_chains: out of memory"); return SER_E_ARG; }
    memcpy(run->h_chain_ids, chain_ids, (size_t)n * sizeof(int));
    CUDA_TRY(POOL_ALLOC(&run->d_chain_ids, (size_t)n * sizeof(int)));
    CUDA_TRY(cudaMemcpyAsync(run->d_chain_ids, chain_ids, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, run->stream));
    CUDA_TRY(cudaStreamSynchronize(run->stream));
    run->kp.chain_ids = run->d_chain_ids;
    return SER_OK;
  };
  if ((rc = attach()) != SER_OK) { ser_run_destroy(run); return rc; }
  *out = run;
  return SER_OK;
}

static size_t acc_bytes(const ser_run *run) { return (size_t)run->cfg.n_chains * acc_layout(run->N, run->M, run->acc_what).ints * sizeof(int); }

/* zero the accumulators of an accumulating run (start of ser_run_init) */
static int acc_zero(ser_run *run)
{
  if (run->d_acc) CUDA_TRY(cudaMemsetAsync(run->d_acc, 0, acc_bytes(run), run->stream));
  return SER_OK;
}

extern "C" int ser_run_accumulate(ser_run *run, int32_t what)
{
  if (!run) { ser_set_error("ser_run_accumulate: null run"); return SER_E_ARG; }
  if (what < 1 || (what & ~SER_ACC_ALL)) { ser_set_error("ser_run_accumulate: bad flags %d", what); return SER_E_ARG; }
  if (run->acc_what) { ser_set_error("ser_run_accumulate: the run already accumulates"); return SER_E_STATE; }
  if (run->sampled) { ser_set_error("ser_run_accumulate: the run has already taken samples; call it before the first sampling call"); return SER_E_STATE; }
  const int need = (what & (SER_ACC_AB | SER_ACC_ALIVE | SER_ACC_RANGE)) ? SER_STORE_FULL : SER_STORE_PI;
  if (run->cfg.store < need) {
    ser_set_error("ser_run_accumulate: these summaries need %s", need == SER_STORE_FULL ? "SER_STORE_FULL (a, b samples)" : "SER_STORE_PI or more");
    return SER_E_STATE;
  }
  if (run->cfg.max_samples < 1) { ser_set_error("ser_run_accumulate: the window needs max_samples >= 1"); return SER_E_ARG; }
  if (set_device(run)) return SER_E_CUDA;
  run->acc_what = what;
  cudaError_t e = POOL_ALLOC(&run->d_acc, acc_bytes(run));
  if (e == cudaSuccess) e = cudaMemsetAsync(run->d_acc, 0, acc_bytes(run), run->stream);
  if (e != cudaSuccess) {
    cudaGetLastError();
    ser_set_error("ser_run_accumulate: cannot allocate %zu bytes of accumulators: %s", acc_bytes(run), cudaGetErrorString(e));
    if (run->d_acc) cudaFreeAsync(run->d_acc, run->stream);
    run->d_acc = nullptr;
    run->acc_what = 0;
    return SER_E_CUDA;
  }
  return SER_OK;
}

extern "C" void ser_run_destroy(ser_run *run)
{
  if (!run) return;
  cudaSetDevice(run->cfg.device);
  void *bufs[] = {run->d_Xs, run->d_hard, run->d_ones, run->d_off, run->d_order, run->d_item_col, run->d_ab, run->d_rpi,
                  run->d_scal, run->d_tape, run->d_tape_off, run->d_samp_a, run->d_samp_b, run->d_samp_pi, run->d_samp_cdl,
                  run->d_scratch_i, run->d_bad, run->d_cd4, run->d_samp_cd_all, run->d_gV, run->d_gpre, run->d_bgrp, run->d_bbat,
                  run->d_V, run->d_queue, run->d_done, run->d_e_all, run->d_info, run->d_chosen, run->d_counts, run->d_unit_tab, run->d_hbits, run->d_col_sites,
                  run->d_chain_ids, run->d_acc};
  for (void *b : bufs) if (b) cudaFreeAsync(b, run->stream);
  if (run->stream) cudaStreamSynchronize(run->stream);
  if (run->sweep_ev) {
    for (cudaEvent_t e : *run->sweep_ev) cudaEventDestroy(e);
    delete run->sweep_ev;
  }
  if (run->ev_start) cudaEventDestroy(run->ev_start);
  if (run->ev_stop) cudaEventDestroy(run->ev_stop);
  if (run->stream) cudaStreamDestroy(run->stream);
  free(run->h_hard);
  free(run->h_chain_ids);
  free(run);
}

extern "C" int ser_run_dims(const ser_run *run, int32_t *N, int32_t *M, int32_t *nh, int32_t *n_chains)
{
  if (!run) return SER_E_ARG;
  if (N) *N = run->N;
  if (M) *M = run->M;
  if (nh) *nh = run->nh;
  if (n_chains) *n_chains = run->cfg.n_chains;
  return SER_OK;
}
extern "C" const uint8_t *ser_run_hard_flags(const ser_run *run) { return run ? run->h_hard : nullptr; }
extern "C" int ser_run_is_manycd(const ser_run *run) { return run ? run->cfg.manycd : 0; }
extern "C" int ser_run_local_chain(const ser_run *run, int32_t g)
{
  if (!run) return -1;
  if (run->h_chain_ids) {
    for (int c = 0; c < run->cfg.n_chains; c++)
      if (run->h_chain_ids[c] == g) return c;
    return -1;
  }
  const int l = g - run->cfg.chain_offset;
  return (l >= 0 && l < run->cfg.n_chains) ? l : -1;
}

extern "C" int ser_run_set_tapes(ser_run *run, const double *flat, const uint64_t *offsets)
{
  if (!run || !flat || !offsets) { ser_set_error("ser_run_set_tapes: null argument"); return SER_E_ARG; }
  if (run->cfg.mode != SER_MODE_REPLAY) { ser_set_error("ser_run_set_tapes: run is not in replay mode"); return SER_E_STATE; }
  if (set_device(run)) return SER_E_CUDA;
  const size_t nc = (size_t)run->cfg.n_chains, total = (size_t)offsets[nc];
  if (run->d_tape) cudaFreeAsync(run->d_tape, run->stream);
  if (run->d_tape_off) cudaFreeAsync(run->d_tape_off, run->stream);
  run->d_tape = nullptr; run->d_tape_off = nullptr;
  CUDA_TRY(POOL_ALLOC(&run->d_tape, (total ? total : 1) * sizeof(double)));
  CUDA_TRY(POOL_ALLOC(&run->d_tape_off, (nc + 1) * sizeof(unsigned long long)));
  CUDA_TRY(cudaMemcpyAsync(run->d_tape, flat, total * sizeof(double), cudaMemcpyHostToDevice, run->stream));
  CUDA_TRY(cudaMemcpyAsync(run->d_tape_off, offsets, (nc + 1) * sizeof(unsigned long long), cudaMemcpyHostToDevice, run->stream));
  CUDA_TRY(cudaStreamSynchronize(run->stream));
  run->kp.tape = run->d_tape; run->kp.tape_off = run->d_tape_off;
  run->have_tapes = 1;
  return SER_OK;
}

extern "C" int ser_run_init(ser_run *run)
{
  if (!run) return SER_E_ARG;
  if (run->cfg.mode == SER_MODE_REPLAY && !run->have_tapes) { ser_set_error("ser_run_init: replay mode needs ser_run_set_tapes first"); return SER_E_TAPE; }
  if (set_device(run)) return SER_E_CUDA;
  if (run->d_done) CUDA_TRY(cudaMemsetAsync(run->d_done, 0, (size_t)run->cfg.n_chains * sizeof(unsigned int), run->stream));
  run->chunks_done = 0;
  if (acc_zero(run)) return SER_E_CUDA;
  run->kp.sample_base = 0;
  run->sampled = 0;
  run->calls_done = 0;
  run->samples_done = 0;
  mark_launch(run);
  ser_init_kernel<<<run->cfg.n_chains, run->Caux, run->smem_init, run->stream>>>(run->kp);
  CUDA_TRY(cudaGetLastError());
  run->initialized = 1;
  return SER_OK;
}

/* One launch = burn_calls burn-in calls, then sample_calls sampling calls, on every chain.
 * One-thread-per-column kernels: a persistent grid (as many CTAs as the device holds) pulls
 * (chain, chunk of calls) work items from a queue, so the last wave of a launch is never longer than
 * one item whatever the number of chains; chunks are as long as the balance allows (>= 32 items per
 * resident CTA when the launch has that much work), because an item boundary costs one state
 * round trip through HBM. */
static int launch_sweeps(ser_run *run, int burn_calls, int sample_calls)
{
  const int n_calls = burn_calls + sample_calls;
  KParams kp = run->kp;
  kp.n_calls = n_calls; kp.burn_calls = burn_calls;
  mark_launch(run);
  /* event pair of this sweep launch */
  if (!run->sweep_ev) run->sweep_ev = new std::vector<cudaEvent_t>();
  const bool rec = run->sweep_ev_used < 2 * 256; /* at most 256 launches between two reads; later ones are not timed */
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  if (rec) {
    if (run->sweep_ev_used + 2 > run->sweep_ev->size()) {
      cudaEvent_t a, b;
      CUDA_TRY(cudaEventCreate(&a)); CUDA_TRY(cudaEventCreate(&b));
      run->sweep_ev->push_back(a); run->sweep_ev->push_back(b);
    }
    ev0 = (*run->sweep_ev)[run->sweep_ev_used]; ev1 = (*run->sweep_ev)[run->sweep_ev_used + 1];
    run->sweep_ev_used += 2;
  }
  int grid = run->sweep_slots; /* large shapes: one CTA per scratch slot, the chains strided over them */
  if (!run->big) {
    const long long work = (long long)run->cfg.n_chains * n_calls;
    int chunk = (int)std::min<long long>(n_calls, std::max<long long>(1, work / (32ll * run->sweep_slots)));
    if (const char *v = getenv("SER_CHUNK_CALLS")) chunk = std::max(1, std::min(n_calls, atoi(v)));
    const int per_chain = (n_calls + chunk - 1) / chunk;
    kp.chunk_calls = chunk;
    kp.n_items = (unsigned int)run->cfg.n_chains * (unsigned int)per_chain;
    kp.chunk_base = run->chunks_done;
    run->chunks_done += (unsigned int)per_chain;
    grid = (int)std::min<long long>((long long)kp.n_items, run->sweep_slots);
    CUDA_TRY(cudaMemsetAsync(run->d_queue, 0, sizeof(unsigned int), run->stream));
  }
  if (rec) CUDA_TRY(cudaEventRecord(ev0, run->stream));
  run->sweep_fn<<<grid, run->sweep_block, run->sweep_smem, run->stream>>>(kp);
  CUDA_TRY(cudaGetLastError());
  if (rec) CUDA_TRY(cudaEventRecord(ev1, run->stream));
  return SER_OK;
}

/* Block shape of a histogram kernel whose threads own rows of `bins` ints (hist_tile): 128 threads, halved down to 32 while their rows
 * do not fit SER_HIST_SMEM bytes of shared memory; rows that do not fit even then are counted in global memory (smem = 0). */
#define SER_HIST_SMEM (96 * 1024)
struct HistShape {
  int threads;
  size_t smem;
};
static cudaError_t hist_shape(const void *kernel, int bins, HistShape *h)
{
  h->threads = 128;
  h->smem = 0;
  while (h->threads > 32 && (size_t)h->threads * bins * sizeof(int) > SER_HIST_SMEM) h->threads >>= 1;
  const size_t bytes = (size_t)h->threads * bins * sizeof(int);
  if (bytes <= SER_HIST_SMEM) h->smem = bytes;
  return h->smem > 48 * 1024 ? cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SER_HIST_SMEM) : cudaSuccess;
}

static PeerPtrs one_dest(void *ptr)
{
  PeerPtrs d;
  memset(&d, 0, sizeof(d));
  d.p[0] = ptr; d.n = 1;
  return d;
}

/* the chosen chains of a getter (d_chosen in the numbering where local chain 0 is id_base); rows as SumSel describes */
static SumSel sel_chosen(const ser_run *run, const int *d_chosen, int id_base, int rows, int *d_n)
{
  return SumSel{d_chosen, id_base, run->cfg.n_chains, run->d_chain_ids, 0, rows, d_n};
}

/* Launches of the summary kernels over k slabs, on the run's stream: the one-shot getters (add = 0) and accumulate_window (add = 1) */
static int launch_po(ser_run *run, const SumSel &sel, int k, const PeerPtrs &dst, size_t stride, int add)
{
  const int N = run->N;
  mark_launch(run);
  ser_po_kernel<<<dim3((N + 31) / 32, (N + 31) / 32, k), 256, 0, run->stream>>>(run->d_samp_pi, run->d_scal, N, run->cfg.max_samples, sel,
                                                                                 dst, stride, add);
  CUDA_TRY(cudaGetLastError());
  return SER_OK;
}

static int launch_posterior(ser_run *run, const SumSel &sel, int k, int *pi, size_t pi_stride, int *a, int *b, size_t ab_stride,
                            long long *corr_num, int add)
{
  mark_launch(run);
  ser_posterior_kernel<<<k, 256, 0, run->stream>>>(run->d_samp_pi, run->d_samp_a, run->d_samp_b, run->d_scal, run->N, run->M,
                                                   run->cfg.max_samples, sel, pi, pi_stride, a, b, ab_stride, corr_num, add);
  CUDA_TRY(cudaGetLastError());
  return SER_OK;
}

static int launch_alive(ser_run *run, const SumSel &sel, int k, int *alive, size_t stride, int add)
{
  mark_launch(run);
  ser_alive_kernel<<<dim3(k, (run->M + 127) / 128), 128, 0, run->stream>>>(run->d_samp_a, run->d_samp_b, run->d_scal, run->N, run->M,
                                                                            run->cfg.max_samples, sel, alive, stride, add);
  CUDA_TRY(cudaGetLastError());
  return SER_OK;
}

static int launch_pos_hist(ser_run *run, const SumSel &sel, int k, int *pos, size_t stride, int add)
{
  const int N = run->N;
  HistShape hs;
  CUDA_TRY(hist_shape((const void *)ser_pos_hist_kernel, N, &hs));
  mark_launch(run);
  ser_pos_hist_kernel<<<dim3(k, (N + hs.threads - 1) / hs.threads), hs.threads, hs.smem, run->stream>>>(
      run->d_samp_pi, run->d_scal, N, run->cfg.max_samples, sel, hs.smem > 0, pos, stride, add);
  CUDA_TRY(cudaGetLastError());
  return SER_OK;
}

static int launch_range_hist(ser_run *run, const SumSel &sel, int k, int *a_hist, int *b_hist, size_t stride, int add)
{
  const int N = run->N, M = run->M;
  HistShape hs;
  CUDA_TRY(hist_shape((const void *)ser_range_hist_kernel, N + 1, &hs));
  mark_launch(run);
  ser_range_hist_kernel<<<dim3(k, (M + hs.threads - 1) / hs.threads, 2), hs.threads, hs.smem, run->stream>>>(
      run->d_samp_a, run->d_samp_b, run->d_scal, N, M, run->cfg.max_samples, sel, hs.smem > 0, a_hist, b_hist, stride, add);
  CUDA_TRY(cudaGetLastError());
  return SER_OK;
}

/* rows [0, w) of every chain's window added into its accumulator record (ser_run_accumulate), on the run's stream */
static int accumulate_window(ser_run *run, int w)
{
  const int what = run->acc_what, nc = run->cfg.n_chains;
  const AccLayout L = acc_layout(run->N, run->M, what);
  const SumSel sel = {nullptr, 0, 0, nullptr, run->kp.sample_base, w, nullptr};
  int *acc = run->d_acc;
  int rc = SER_OK;
  if (what & SER_ACC_PO) rc = launch_po(run, sel, nc, one_dest(acc + L.po), L.ints, 1);
  if (!rc && (what & (SER_ACC_SUMS | SER_ACC_AB))) {
    const bool ab = what & SER_ACC_AB;
    rc = launch_posterior(run, sel, nc, acc + L.pi, L.ints, ab ? acc + L.asum : nullptr, ab ? acc + L.bsum : nullptr, L.ints, nullptr, 1);
  }
  if (!rc && (what & SER_ACC_ALIVE)) rc = launch_alive(run, sel, nc, acc + L.alive, L.ints, 1);
  if (!rc && (what & SER_ACC_POS)) rc = launch_pos_hist(run, sel, nc, acc + L.pos, L.ints, 1);
  if (!rc && (what & SER_ACC_RANGE)) rc = launch_range_hist(run, sel, nc, acc + L.range, acc + L.range + (size_t)run->M * (run->N + 1), L.ints, 1);
  return rc;
}

extern "C" int ser_run_advance_both(ser_run *run, int32_t burn_calls, int32_t sample_calls)
{
  if (!run) return SER_E_ARG;
  if (!run->initialized) { ser_set_error("ser_run_advance: call ser_run_init first"); return SER_E_STATE; }
  if (burn_calls < 0 || sample_calls < 0) { ser_set_error("ser_run_advance: negative call count"); return SER_E_ARG; }
  if (burn_calls + sample_calls <= 0) return SER_OK;
  if (set_device(run)) return SER_E_CUDA;
  if (sample_calls > 0) run->sampled = 1;
  run->calls_done += burn_calls + sample_calls;
  run->samples_done += sample_calls;
  if (!run->acc_what) return launch_sweeps(run, burn_calls, sample_calls);
  /* accumulating run: launches of at most one window of sampling calls (the burn-in rides on the first), each followed by the
   * accumulation of the rows it wrote; splitting a launch changes no chain */
  do {
    const int w = std::min(sample_calls, run->cfg.max_samples);
    int rc = launch_sweeps(run, burn_calls, w);
    if (rc == SER_OK && w > 0) rc = accumulate_window(run, w);
    if (rc != SER_OK) return rc;
    run->kp.sample_base += w;
    burn_calls = 0;
    sample_calls -= w;
  } while (sample_calls > 0);
  return SER_OK;
}

/* total CUDA-event time of the sweep launches since the last reset and their number (waits for the last one) */
extern "C" int ser_run_sweep_time(ser_run *run, double *ms, int32_t *n_launches, int32_t reset)
{
  if (!run || !ms) return SER_E_ARG;
  if (set_device(run)) return SER_E_CUDA;
  double total = 0.0;
  for (size_t i = 0; i + 1 < run->sweep_ev_used; i += 2) {
    float t = 0.f;
    CUDA_TRY(cudaEventSynchronize((*run->sweep_ev)[i + 1]));
    CUDA_TRY(cudaEventElapsedTime(&t, (*run->sweep_ev)[i], (*run->sweep_ev)[i + 1]));
    total += t;
  }
  *ms = total;
  if (n_launches) *n_launches = (int32_t)(run->sweep_ev_used / 2);
  if (reset) run->sweep_ev_used = 0;
  return SER_OK;
}

extern "C" int ser_run_advance(ser_run *run, int32_t n_calls, int32_t sampling)
{
  return sampling ? ser_run_advance_both(run, 0, n_calls) : ser_run_advance_both(run, n_calls, 0);
}

extern "C" int ser_run_sync(ser_run *run)
{
  if (!run) return SER_E_ARG;
  if (set_device(run)) return SER_E_CUDA;
  CUDA_TRY(cudaStreamSynchronize(run->stream));
  return SER_OK;
}

extern "C" int ser_run_elapsed_ms(ser_run *run, double *ms, int32_t reset)
{
  if (!run || !ms) return SER_E_ARG;
  if (set_device(run)) return SER_E_CUDA;
  if (run->timing_open) {
    CUDA_TRY(cudaEventRecord(run->ev_stop, run->stream));
    CUDA_TRY(cudaEventSynchronize(run->ev_stop));
    float t = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&t, run->ev_start, run->ev_stop));
    run->elapsed_ms += t;
    run->timing_open = 0;
  }
  *ms = run->elapsed_ms;
  if (reset) run->elapsed_ms = 0.0;
  return SER_OK;
}

extern "C" int ser_run_kernel_launches(const ser_run *run, int64_t *n)
{
  if (!run || !n) return SER_E_ARG;
  *n = run->launches;
  return SER_OK;
}

extern "C" int ser_run_kernel_path(const ser_run *run, int32_t *path)
{
  if (!run || !path) return SER_E_ARG;
  *path = !run->big ? 0 : run->big_warp ? 2 : 1;
  return SER_OK;
}

static int chain_ok(ser_run *run, int chain)
{
  if (!run) { ser_set_error("null run"); return 0; }
  if (chain < 0 || chain >= run->cfg.n_chains) { ser_set_error("chain %d out of range [0,%d)", chain, run->cfg.n_chains); return 0; }
  return 1;
}

extern "C" int ser_run_get_state(ser_run *run, int32_t chain, int32_t *a, int32_t *b, int32_t *pi, int32_t *rpi, int32_t *t0,
                                 int32_t *f0, int32_t *t1, int32_t *f1, int32_t tot[4], double cdl[3], int64_t *tape_slots)
{
  if (!chain_ok(run, chain)) return SER_E_ARG;
  if (!run->initialized) { ser_set_error("ser_run_get_state: run not initialised"); return SER_E_STATE; }
  if (set_device(run)) return SER_E_CUDA;
  const int N = run->N, M = run->M;
  int *d = run->d_scratch_i;
  int *d_a = d, *d_b = d + M, *d_pi = d + 2 * M, *d_rpi = d + 2 * M + N, *d_cnt = d + 2 * M + 2 * N;
  mark_launch(run);
  ser_export_kernel<<<1, run->Caux, run->smem_small, run->stream>>>(run->kp, chain, d_a, d_b, d_pi, d_rpi, d_cnt);
  CUDA_TRY(cudaGetLastError());
  std::vector<int> h(2 * N + 6 * M);
  ChainScalars sc;
  CUDA_TRY(cudaMemcpyAsync(h.data(), d, h.size() * sizeof(int), cudaMemcpyDeviceToHost, run->stream));
  CUDA_TRY(cudaMemcpyAsync(&sc, run->d_scal + chain, sizeof(sc), cudaMemcpyDeviceToHost, run->stream));
  CUDA_TRY(cudaStreamSynchronize(run->stream));
  if (a) memcpy(a, h.data(), M * 4);
  if (b) memcpy(b, h.data() + M, M * 4);
  if (pi) memcpy(pi, h.data() + 2 * M, N * 4);
  if (rpi) memcpy(rpi, h.data() + 2 * M + N, N * 4);
  const int *cnt = h.data() + 2 * M + 2 * N;
  if (t0) memcpy(t0, cnt, M * 4);
  if (f0) memcpy(f0, cnt + M, M * 4);
  if (t1) memcpy(t1, cnt + 2 * M, M * 4);
  if (f1) memcpy(f1, cnt + 3 * M, M * 4);
  if (tot) { tot[0] = sc.t0a; tot[1] = sc.f0a; tot[2] = sc.t1a; tot[3] = sc.f1a; }
  if (cdl) { cdl[0] = sc.c; cdl[1] = sc.d; cdl[2] = sc.loglik; }
  if (tape_slots) *tape_slots = sc.cursor;
  if (sc.flags & 1) { ser_set_error("chain %d: replay tape exhausted", chain); return SER_E_TAPE; }
  return SER_OK;
}

extern "C" int ser_run_get_counters(ser_run *run, int32_t chain, int64_t out[8])
{
  if (!chain_ok(run, chain) || !out) return SER_E_ARG;
  if (set_device(run)) return SER_E_CUDA;
  ChainScalars sc;
  CUDA_TRY(cudaMemcpyAsync(&sc, run->d_scal + chain, sizeof(sc), cudaMemcpyDeviceToHost, run->stream));
  CUDA_TRY(cudaStreamSynchronize(run->stream));
  for (int i = 0; i < 8; i++) out[i] = sc.counters[i];
  return SER_OK;
}

/* flags of one chain after ser_run_check: 1 tape exhausted, 2 a/b range, 4 permutation, 8 hard-site order, 16 totals / loglik */
extern "C" int ser_run_get_flags(ser_run *run, int32_t chain, int32_t *flags)
{
  if (!chain_ok(run, chain) || !flags) return SER_E_ARG;
  if (set_device(run)) return SER_E_CUDA;
  ChainScalars sc;
  CUDA_TRY(cudaMemcpyAsync(&sc, run->d_scal + chain, sizeof(sc), cudaMemcpyDeviceToHost, run->stream));
  CUDA_TRY(cudaStreamSynchronize(run->stream));
  *flags = sc.flags & 31; /* bit 5 is internal (bit columns stored) */
  return SER_OK;
}

extern "C" int ser_run_check(ser_run *run, int32_t *n_bad)
{
  if (!run || !n_bad) return SER_E_ARG;
  if (!run->initialized) { ser_set_error("ser_run_check: run not initialised"); return SER_E_STATE; }
  if (set_device(run)) return SER_E_CUDA;
  CUDA_TRY(cudaMemsetAsync(run->d_bad, 0, sizeof(int), run->stream));
  mark_launch(run);
  ser_check_kernel<<<run->cfg.n_chains, run->Caux, run->smem_small, run->stream>>>(run->kp, run->d_bad);
  CUDA_TRY(cudaGetLastError());
  int bad = 0;
  CUDA_TRY(cudaMemcpyAsync(&bad, run->d_bad, sizeof(int), cudaMemcpyDeviceToHost, run->stream));
  CUDA_TRY(cudaStreamSynchronize(run->stream));
  *n_bad = bad;
  if (bad) { ser_set_error("ser_run_check: %d inconsistent chain(s)", bad); return SER_E_CHECK; }
  return SER_OK;
}

extern "C" int ser_run_chain_sums(ser_run *run, int32_t chain, double sums[3], int32_t *n_samples)
{
  if (!chain_ok(run, chain)) return SER_E_ARG;
  if (set_device(run)) return SER_E_CUDA;
  ChainScalars sc;
  CUDA_TRY(cudaMemcpyAsync(&sc, run->d_scal + chain, sizeof(sc), cudaMemcpyDeviceToHost, run->stream));
  CUDA_TRY(cudaStreamSynchronize(run->stream));
  if (sums) { sums[0] = sc.sum_negll; sums[1] = sc.sum_ec; sums[2] = sc.sum_ed; }
  if (n_samples) *n_samples = sc.n_samples;
  return SER_OK;
}

extern "C" int ser_run_chain_stats(ser_run *run, double *e_negloglik, double *e_c, double *e_d, int32_t *n_samples)
{
  if (!run) return SER_E_ARG;
  if (set_device(run)) return SER_E_CUDA;
  const int nc = run->cfg.n_chains;
  std::vector<ChainScalars> sc(nc);
  CUDA_TRY(cudaMemcpyAsync(sc.data(), run->d_scal, (size_t)nc * sizeof(ChainScalars), cudaMemcpyDeviceToHost, run->stream));
  CUDA_TRY(cudaStreamSynchronize(run->stream));
  for (int i = 0; i < nc; i++) {
    const double n = sc[i].n_samples > 0 ? (double)sc[i].n_samples : 1.0;
    if (e_negloglik) e_negloglik[i] = sc[i].sum_negll / n;
    if (e_c) e_c[i] = sc[i].sum_ec / n;
    if (e_d) e_d[i] = sc[i].sum_ed / n;
  }
  if (n_samples) *n_samples = sc[0].n_samples;
  return SER_OK;
}

/* E[-logL] of the local chains at dst[offset + chain] of every destination, on the run's stream */
static int run_stats_to(ser_run *run, const PeerPtrs &dst, int offset)
{
  const int nc = run->cfg.n_chains;
  mark_launch(run);
  ser_stats_kernel<<<(nc + 255) / 256, 256, 0, run->stream>>>(run->d_scal, nc, dst, offset);
  CUDA_TRY(cudaGetLastError());
  return SER_OK;
}

/* pair-order slabs of the chosen chains this run owns, into every destination, on the run's stream */
/* id_base = the id local chain 0 has in the numbering `d_chosen` uses */
static int run_po_to(ser_run *run, const int32_t *d_chosen, int k, const PeerPtrs &dst, int id_base)
{
  return launch_po(run, sel_chosen(run, d_chosen, id_base, run->cfg.max_samples, nullptr), k, dst, (size_t)run->N * run->N, 0);
}

extern "C" int ser_run_chain_stats_device(ser_run *run, double *d_e_negloglik)
{
  if (!run || !d_e_negloglik) return SER_E_ARG;
  if (set_device(run)) return SER_E_CUDA;
  return run_stats_to(run, one_dest(d_e_negloglik), 0);
}

extern "C" int ser_run_fetch_samples(ser_run *run, int32_t chain, int32_t *a, int32_t *b, int32_t *pi, double *c, double *d,
                                     double *loglik, int32_t *n)
{
  if (!chain_ok(run, chain)) return SER_E_ARG;
  if (run->acc_what) { ser_set_error("ser_run_fetch_samples: the store of an accumulating run is a transient window; read the summaries"); return SER_E_STATE; }
  if (set_device(run)) return SER_E_CUDA;
  ChainScalars sc;
  CUDA_TRY(cudaMemcpyAsync(&sc, run->d_scal + chain, sizeof(sc), cudaMemcpyDeviceToHost, run->stream));
  CUDA_TRY(cudaStreamSynchronize(run->stream));
  const int ns = sc.n_samples < run->cfg.max_samples ? sc.n_samples : run->cfg.max_samples;
  if (n) *n = ns;
  const int N = run->N, M = run->M;
  const size_t row0 = (size_t)chain * run->cfg.max_samples;
  if ((a || b || c || d || loglik) && run->cfg.store < SER_STORE_FULL) { ser_set_error("ser_run_fetch_samples: run was created without SER_STORE_FULL"); return SER_E_STATE; }
  if (pi && run->cfg.store < SER_STORE_PI) { ser_set_error("ser_run_fetch_samples: run was created without a sample store"); return SER_E_STATE; }
  std::vector<uint16_t> tmp;
  auto fetch16 = [&](const uint16_t *src, int width, int32_t *dst) -> int {
    tmp.resize((size_t)ns * width);
    if (cudaMemcpyAsync(tmp.data(), src + row0 * width, tmp.size() * 2, cudaMemcpyDeviceToHost, run->stream) != cudaSuccess) return 1;
    if (cudaStreamSynchronize(run->stream) != cudaSuccess) return 1;
    for (size_t i = 0; i < tmp.size(); i++) dst[i] = tmp[i];
    return 0;
  };
  if (ns > 0) {
    if (a && fetch16(run->d_samp_a, M, a)) { ser_set_error("fetch a failed"); return SER_E_CUDA; }
    if (b && fetch16(run->d_samp_b, M, b)) { ser_set_error("fetch b failed"); return SER_E_CUDA; }
    if (pi && fetch16(run->d_samp_pi, N, pi)) { ser_set_error("fetch pi failed"); return SER_E_CUDA; }
    if (c || d || loglik) {
      std::vector<double> cdl((size_t)ns * 3);
      CUDA_TRY(cudaMemcpyAsync(cdl.data(), run->d_samp_cdl + row0 * 3, cdl.size() * 8, cudaMemcpyDeviceToHost, run->stream));
      CUDA_TRY(cudaStreamSynchronize(run->stream));
      for (int s = 0; s < ns; s++) {
        if (c) c[s] = cdl[3 * s];
        if (d) d[s] = cdl[3 * s + 1];
        if (loglik) loglik[s] = cdl[3 * s + 2];
      }
    }
  }
  return SER_OK;
}

/* manycd runs: per-taxon c, d of one chain (file order) */
extern "C" int ser_run_get_cd(ser_run *run, int32_t chain, double *c, double *d)
{
  if (!chain_ok(run, chain)) return SER_E_ARG;
  if (!run->cfg.manycd) { ser_set_error("ser_run_get_cd: run was created with manycd = 0"); return SER_E_STATE; }
  if (!run->initialized) { ser_set_error("ser_run_get_cd: run not initialised"); return SER_E_STATE; }
  if (set_device(run)) return SER_E_CUDA;
  const int M = run->M, Mpad = run->kp.Mpad;
  std::vector<double> h((size_t)4 * Mpad);
  std::vector<uint16_t> order(M);
  CUDA_TRY(cudaMemcpyAsync(h.data(), run->d_cd4 + (size_t)chain * 4 * Mpad, h.size() * 8, cudaMemcpyDeviceToHost, run->stream));
  CUDA_TRY(cudaMemcpyAsync(order.data(), run->d_order, M * sizeof(uint16_t), cudaMemcpyDeviceToHost, run->stream));
  CUDA_TRY(cudaStreamSynchronize(run->stream));
  for (int col = 0; col < M; col++) {
    if (c) c[order[col]] = h[col];
    if (d) d[order[col]] = h[2 * Mpad + col];
  }
  return SER_OK;
}

/* manycd runs with SER_STORE_FULL: per-taxon c, d of every stored sample, [n][M] each */
extern "C" int ser_run_fetch_cd_samples(ser_run *run, int32_t chain, double *c, double *d, int32_t *n)
{
  if (!chain_ok(run, chain)) return SER_E_ARG;
  if (!run->cfg.manycd || !run->d_samp_cd_all) { ser_set_error("ser_run_fetch_cd_samples: needs manycd = 1 and SER_STORE_FULL"); return SER_E_STATE; }
  if (run->acc_what) { ser_set_error("ser_run_fetch_cd_samples: the store of an accumulating run is a transient window"); return SER_E_STATE; }
  if (set_device(run)) return SER_E_CUDA;
  ChainScalars sc;
  CUDA_TRY(cudaMemcpyAsync(&sc, run->d_scal + chain, sizeof(sc), cudaMemcpyDeviceToHost, run->stream));
  CUDA_TRY(cudaStreamSynchronize(run->stream));
  const int ns = sc.n_samples < run->cfg.max_samples ? sc.n_samples : run->cfg.max_samples, M = run->M;
  if (n) *n = ns;
  if (ns > 0 && (c || d)) {
    std::vector<double> h((size_t)ns * 2 * M);
    CUDA_TRY(cudaMemcpyAsync(h.data(), run->d_samp_cd_all + (size_t)chain * run->cfg.max_samples * 2 * M, h.size() * 8,
                             cudaMemcpyDeviceToHost, run->stream));
    CUDA_TRY(cudaStreamSynchronize(run->stream));
    for (int s = 0; s < ns; s++) {
      if (c) memcpy(c + (size_t)s * M, h.data() + ((size_t)s * 2 + 0) * M, M * 8);
      if (d) memcpy(d + (size_t)s * M, h.data() + ((size_t)s * 2 + 1) * M, M * 8);
    }
  }
  return SER_OK;
}

extern "C" int ser_select_chains_device(const double *d_e, int32_t n, int32_t k, int32_t *d_chosen, double *d_info, int32_t device,
                                        void *stream)
{
  if (!d_e || !d_chosen || !d_info || n < 1 || k < 1) { ser_set_error("ser_select_chains_device: bad argument"); return SER_E_ARG; }
  CUDA_TRY(cudaSetDevice(device));
  ser_select_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(d_e, n, k, d_chosen, d_info);
  CUDA_TRY(cudaGetLastError());
  return SER_OK;
}

/* d_counts [k][N][N]; n_out[c] = T of a held chain when d_n is given */
static int po_counts_to(ser_run *run, const int32_t *d_chosen, int k, int32_t *d_counts, int *d_n)
{
  if (run->cfg.store < SER_STORE_PI) { ser_set_error("ser_run_po_counts: run has no pi sample store"); return SER_E_STATE; }
  if (!run->acc_what) /* T is read per chosen chain on the device: no host round trip */
    return launch_po(run, sel_chosen(run, d_chosen, run->cfg.chain_offset, run->cfg.max_samples, d_n), k, one_dest(d_counts),
                     (size_t)run->N * run->N, 0);
  if (!(run->acc_what & SER_ACC_PO)) { ser_set_error("ser_run_po_counts: the run accumulates without SER_ACC_PO"); return SER_E_STATE; }
  const int N = run->N, nb = (int)std::min<long long>(((long long)N * N + 255) / 256, 1024);
  const AccLayout L = acc_layout(N, run->M, run->acc_what);
  mark_launch(run);
  ser_po_acc_out_kernel<<<dim3(nb, k), 256, 0, run->stream>>>(run->d_acc + L.po, L.ints, run->d_scal, N,
                                                              sel_chosen(run, d_chosen, run->cfg.chain_offset, INT_MAX, d_n), d_counts);
  CUDA_TRY(cudaGetLastError());
  return SER_OK;
}

extern "C" int ser_run_po_counts_device(ser_run *run, const int32_t *d_chosen, int32_t k, int32_t *d_counts)
{
  if (!run || !d_chosen || !d_counts || k < 1) return SER_E_ARG;
  if (set_device(run)) return SER_E_CUDA;
  return po_counts_to(run, d_chosen, k, d_counts, nullptr);
}

/* One host output of a getter: k slabs of `bytes` each at `host` (nullptr: not wanted), staged through `dev`. */
struct GetterOut {
  void *host;
  size_t bytes;
  void *dev;
};

/* The shared part of the host getters over k chosen global ids: the ids go up, n_out[c] starts at -1 and `launch` (given the device
 * ids and n_out) enqueues kernels that write T and the slabs of every chosen chain the run holds; those slabs come back to the host,
 * the others stay as the caller passed them.  Every temporary is freed on every path. */
template <class Launch>
static int run_getter(ser_run *run, const int32_t *chosen, int k, std::vector<int> &n_out, std::initializer_list<GetterOut *> outs,
                      Launch launch)
{
  int *d_ch = nullptr, *d_n = nullptr;
  n_out.assign(k, -1);
  auto body = [&]() -> int {
    CUDA_TRY(POOL_ALLOC(&d_ch, k * sizeof(int)));
    CUDA_TRY(POOL_ALLOC(&d_n, k * sizeof(int)));
    for (GetterOut *o : outs)
      if (o->host) CUDA_TRY(POOL_ALLOC(&o->dev, k * o->bytes));
    CUDA_TRY(cudaMemcpyAsync(d_ch, chosen, k * sizeof(int), cudaMemcpyHostToDevice, run->stream));
    CUDA_TRY(cudaMemsetAsync(d_n, 0xff, k * sizeof(int), run->stream));
    const int rc = launch(d_ch, d_n);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(n_out.data(), d_n, k * sizeof(int), cudaMemcpyDeviceToHost, run->stream));
    CUDA_TRY(cudaStreamSynchronize(run->stream));
    for (int c = 0; c < k; c++)
      for (GetterOut *o : outs)
        if (o->host && n_out[c] >= 0)
          CUDA_TRY(cudaMemcpyAsync((char *)o->host + c * o->bytes, (char *)o->dev + c * o->bytes, o->bytes, cudaMemcpyDeviceToHost, run->stream));
    CUDA_TRY(cudaStreamSynchronize(run->stream));
    return SER_OK;
  };
  const int rc = body();
  if (d_ch) cudaFreeAsync(d_ch, run->stream);
  if (d_n) cudaFreeAsync(d_n, run->stream);
  for (GetterOut *o : outs)
    if (o->dev) { cudaFreeAsync(o->dev, run->stream); o->dev = nullptr; }
  return rc;
}

extern "C" int ser_run_po_counts(ser_run *run, const int32_t *chosen, int32_t k, int32_t *counts)
{
  if (!run || !chosen || !counts || k < 1) return SER_E_ARG;
  if (set_device(run)) return SER_E_CUDA;
  GetterOut cnt = {counts, (size_t)run->N * run->N * sizeof(int), nullptr};
  std::vector<int> n_out;
  return run_getter(run, chosen, k, n_out, {&cnt}, [&](const int *d_ch, int *d_n) { return po_counts_to(run, d_ch, k, (int *)cnt.dev, d_n); });
}

/* common sample count of the chosen chains this run owns (n_out[c] < 0: not owned) */
static int common_samples(const std::vector<int> &n_out, int32_t *n_samples, const char *who)
{
  int ns = -1;
  for (int v : n_out) {
    if (v < 0) continue;
    if (ns >= 0 && v != ns) { ser_set_error("%s: the chosen chains hold different numbers of samples (%d vs %d)", who, ns, v); return SER_E_STATE; }
    ns = v;
  }
  if (n_samples) *n_samples = ns < 0 ? 0 : ns;
  return SER_OK;
}

extern "C" int ser_run_posterior_sums(ser_run *run, const int32_t *chosen, int32_t k, int64_t *corr_num, int32_t *pi_sum,
                                      int32_t *a_sum, int32_t *b_sum, int32_t *n_samples)
{
  if (!run || !chosen || !corr_num || !pi_sum || k < 1) { ser_set_error("ser_run_posterior_sums: bad argument"); return SER_E_ARG; }
  if (run->cfg.store < SER_STORE_PI) { ser_set_error("ser_run_posterior_sums: run has no pi sample store"); return SER_E_STATE; }
  if ((a_sum || b_sum) && run->cfg.store < SER_STORE_FULL) { ser_set_error("ser_run_posterior_sums: a/b sums need SER_STORE_FULL"); return SER_E_STATE; }
  if (run->acc_what && !(run->acc_what & SER_ACC_SUMS)) { ser_set_error("ser_run_posterior_sums: the run accumulates without SER_ACC_SUMS"); return SER_E_STATE; }
  if (run->acc_what && (a_sum || b_sum) && !(run->acc_what & SER_ACC_AB)) { ser_set_error("ser_run_posterior_sums: the run accumulates without SER_ACC_AB"); return SER_E_STATE; }
  if (set_device(run)) return SER_E_CUDA;
  const int N = run->N, M = run->M;
  GetterOut corr = {corr_num, sizeof(long long), nullptr}, pi = {pi_sum, N * sizeof(int), nullptr};
  GetterOut a = {a_sum, M * sizeof(int), nullptr}, b = {b_sum, M * sizeof(int), nullptr};
  std::vector<int> n_out;
  const int rc = run_getter(run, chosen, k, n_out, {&corr, &pi, &a, &b}, [&](const int *d_ch, int *d_n) -> int {
    if (!run->acc_what)
      return launch_posterior(run, sel_chosen(run, d_ch, run->cfg.chain_offset, run->cfg.max_samples, d_n), k, (int *)pi.dev, N,
                              (int *)a.dev, (int *)b.dev, M, (long long *)corr.dev, 0);
    const AccLayout L = acc_layout(N, M, run->acc_what);
    mark_launch(run);
    ser_posterior_acc_out_kernel<<<k, 256, 0, run->stream>>>(run->d_acc + L.pi, run->d_acc + L.asum, run->d_acc + L.bsum, L.ints, run->d_scal,
                                                             N, M, sel_chosen(run, d_ch, run->cfg.chain_offset, INT_MAX, d_n),
                                                             (long long *)corr.dev, (int *)pi.dev, (int *)a.dev, (int *)b.dev);
    CUDA_TRY(cudaGetLastError());
    return SER_OK;
  });
  if (rc != SER_OK) return rc;
  return common_samples(n_out, n_samples, "ser_run_posterior_sums");
}

extern "C" int ser_run_alive_counts(ser_run *run, const int32_t *chosen, int32_t k, int32_t *alive, int32_t *n_samples)
{
  if (!run || !chosen || !alive || k < 1) { ser_set_error("ser_run_alive_counts: bad argument"); return SER_E_ARG; }
  if (run->cfg.store < SER_STORE_FULL) { ser_set_error("ser_run_alive_counts: needs SER_STORE_FULL (a, b samples)"); return SER_E_STATE; }
  if (run->acc_what && !(run->acc_what & SER_ACC_ALIVE)) { ser_set_error("ser_run_alive_counts: the run accumulates without SER_ACC_ALIVE"); return SER_E_STATE; }
  if (set_device(run)) return SER_E_CUDA;
  const int N = run->N, M = run->M;
  GetterOut out = {alive, (size_t)N * M * sizeof(int), nullptr};
  std::vector<int> n_out;
  const int rc = run_getter(run, chosen, k, n_out, {&out}, [&](const int *d_ch, int *d_n) -> int {
    if (!run->acc_what)
      return launch_alive(run, sel_chosen(run, d_ch, run->cfg.chain_offset, run->cfg.max_samples, d_n), k, (int *)out.dev, (size_t)N * M, 0);
    const AccLayout L = acc_layout(N, M, run->acc_what);
    mark_launch(run);
    ser_alive_acc_out_kernel<<<dim3(k, (M + 127) / 128), 128, 0, run->stream>>>(run->d_acc + L.alive, L.ints, run->d_scal, N, M,
                                                                                 sel_chosen(run, d_ch, run->cfg.chain_offset, INT_MAX, d_n),
                                                                                 (int *)out.dev);
    CUDA_TRY(cudaGetLastError());
    return SER_OK;
  });
  if (rc != SER_OK) return rc;
  return common_samples(n_out, n_samples, "ser_run_alive_counts");
}

extern "C" int ser_run_marginals(ser_run *run, const int32_t *chosen, int32_t k, int32_t *pos, int32_t *a_hist, int32_t *b_hist,
                                 int32_t *n_samples)
{
  if (!run || !chosen || !n_samples || k < 1 || (!pos && !a_hist && !b_hist)) {
    ser_set_error("ser_run_marginals: bad argument (k = %d; chosen, n_samples and at least one of pos, a_hist, b_hist are needed)", k);
    return SER_E_ARG;
  }
  if (!run->initialized) { ser_set_error("ser_run_marginals: run not initialised"); return SER_E_STATE; }
  const bool ranges = a_hist || b_hist;
  if (pos && run->cfg.store < SER_STORE_PI) { ser_set_error("ser_run_marginals: positions need SER_STORE_PI"); return SER_E_STATE; }
  if (ranges && run->cfg.store < SER_STORE_FULL) { ser_set_error("ser_run_marginals: a / b histograms need SER_STORE_FULL"); return SER_E_STATE; }
  if (run->acc_what && pos && !(run->acc_what & SER_ACC_POS)) { ser_set_error("ser_run_marginals: the run accumulates without SER_ACC_POS"); return SER_E_STATE; }
  if (run->acc_what && ranges && !(run->acc_what & SER_ACC_RANGE)) {
    ser_set_error("ser_run_marginals: the run accumulates without SER_ACC_RANGE");
    return SER_E_STATE;
  }
  if (set_device(run)) return SER_E_CUDA;
  const int N = run->N, M = run->M;
  const size_t pos_cells = (size_t)N * N, range_cells = (size_t)M * (N + 1);
  GetterOut p = {pos, pos_cells * sizeof(int), nullptr}, a = {a_hist, range_cells * sizeof(int), nullptr}, b = {b_hist, range_cells * sizeof(int), nullptr};
  std::vector<int> n_out;
  const int rc = run_getter(run, chosen, k, n_out, {&p, &a, &b}, [&](const int *d_ch, int *d_n) -> int {
    if (!run->acc_what) {
      const SumSel sel = sel_chosen(run, d_ch, run->cfg.chain_offset, run->cfg.max_samples, d_n);
      int rc = pos ? launch_pos_hist(run, sel, k, (int *)p.dev, pos_cells, 0) : SER_OK;
      if (!rc && ranges) rc = launch_range_hist(run, sel, k, (int *)a.dev, (int *)b.dev, range_cells, 0);
      return rc;
    }
    const AccLayout L = acc_layout(N, M, run->acc_what);
    const SumSel sel = sel_chosen(run, d_ch, run->cfg.chain_offset, INT_MAX, d_n);
    if (pos) {
      mark_launch(run);
      ser_hist_acc_out_kernel<<<dim3(256, k, 1), 256, 0, run->stream>>>(run->d_acc + L.pos, L.ints, pos_cells, run->d_scal, sel, (int *)p.dev, nullptr);
      CUDA_TRY(cudaGetLastError());
    }
    if (ranges) {
      mark_launch(run);
      ser_hist_acc_out_kernel<<<dim3(256, k, 2), 256, 0, run->stream>>>(run->d_acc + L.range, L.ints, range_cells, run->d_scal, sel, (int *)a.dev,
                                                                        (int *)b.dev);
      CUDA_TRY(cudaGetLastError());
    }
    return SER_OK;
  });
  if (rc != SER_OK) return rc;
  for (int c = 0; c < k; c++) n_samples[c] = n_out[c] < 0 ? 0 : n_out[c];
  return SER_OK;
}

extern "C" int ser_run_diagnostics(ser_run *run, const int32_t *chosen, int32_t k, int32_t what, int32_t max_lag, double *stats,
                                   double *halves, int32_t *n_samples)
{
  if (!run || !chosen || !stats || !halves || !n_samples || k < 1 || what < 1 || what > 3 || max_lag < 0) {
    ser_set_error("ser_run_diagnostics: bad argument (k = %d, what = %d, max_lag = %d)", k, what, max_lag);
    return SER_E_ARG;
  }
  if (!run->initialized) { ser_set_error("ser_run_diagnostics: run not initialised"); return SER_E_STATE; }
  if (run->acc_what) { ser_set_error("ser_run_diagnostics: the store of an accumulating run is a transient window"); return SER_E_STATE; }
  if ((what & SER_DIAG_SCALARS) && run->cfg.store < SER_STORE_FULL) {
    ser_set_error("ser_run_diagnostics: -loglik, exp(c), exp(d) need SER_STORE_FULL");
    return SER_E_STATE;
  }
  if ((what & SER_DIAG_SITES) && run->cfg.store < SER_STORE_PI) { ser_set_error("ser_run_diagnostics: pi needs SER_STORE_PI"); return SER_E_STATE; }
  if (set_device(run)) return SER_E_CUDA;
  const int Q = 3 + run->N, qlo = (what & SER_DIAG_SCALARS) ? 0 : 3, qhi = (what & SER_DIAG_SITES) ? Q : 3;
  const size_t cells = (size_t)k * Q * 4;
  int *d_ch = nullptr, *d_n = nullptr;
  double *d_stats = nullptr, *d_halves = nullptr;
  std::vector<int> n_out(k);
  auto body = [&]() -> int {
    CUDA_TRY(POOL_ALLOC(&d_ch, k * sizeof(int)));
    CUDA_TRY(POOL_ALLOC(&d_n, k * sizeof(int)));
    CUDA_TRY(POOL_ALLOC(&d_stats, cells * sizeof(double)));
    CUDA_TRY(POOL_ALLOC(&d_halves, cells * sizeof(double)));
    CUDA_TRY(cudaMemcpyAsync(d_ch, chosen, k * sizeof(int), cudaMemcpyHostToDevice, run->stream));
    CUDA_TRY(cudaMemsetAsync(d_n, 0xff, k * sizeof(int), run->stream));
    CUDA_TRY(cudaMemcpyAsync(d_stats, stats, cells * sizeof(double), cudaMemcpyHostToDevice, run->stream));
    CUDA_TRY(cudaMemcpyAsync(d_halves, halves, cells * sizeof(double), cudaMemcpyHostToDevice, run->stream));
    mark_launch(run);
    ser_diag_kernel<<<dim3(k, (qhi - 1) / 32 - qlo / 32 + 1), 1024, 0, run->stream>>>(
        run->d_samp_pi, run->d_samp_cdl, run->d_scal, run->N, run->cfg.max_samples, d_ch, run->cfg.chain_offset, run->cfg.n_chains,
        run->d_chain_ids, qlo, qhi, max_lag, d_stats, d_halves, d_n);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(n_out.data(), d_n, k * sizeof(int), cudaMemcpyDeviceToHost, run->stream));
    CUDA_TRY(cudaStreamSynchronize(run->stream));
    for (int c = 0; c < k; c++)
      if (n_out[c] >= 0 && n_out[c] < 4) {
        ser_set_error("ser_run_diagnostics: chain %d holds %d stored samples (at least 4 are needed)", chosen[c], n_out[c]);
        return SER_E_STATE;
      }
    CUDA_TRY(cudaMemcpyAsync(stats, d_stats, cells * sizeof(double), cudaMemcpyDeviceToHost, run->stream));
    CUDA_TRY(cudaMemcpyAsync(halves, d_halves, cells * sizeof(double), cudaMemcpyDeviceToHost, run->stream));
    CUDA_TRY(cudaStreamSynchronize(run->stream));
    for (int c = 0; c < k; c++)
      if (n_out[c] >= 0) n_samples[c] = n_out[c];
    return SER_OK;
  };
  const int rc = body();
  void *tmp[] = {d_ch, d_n, d_stats, d_halves};
  for (void *t : tmp) if (t) cudaFreeAsync(t, run->stream);
  return rc;
}

/* ------------------------------------------------------------------ the cross-chain step on one stream
 * stats -> (all-gather) -> selection -> zero counts -> pair-order slabs -> (all-reduce): six enqueues, no host
 * synchronisation (script.py:70-99 + :155-189 over run_all_chains' chains, :48-67). */
extern "C" int ser_run_cross_chain_async(ser_run *run, ser_comm *comm, int32_t k)
{
  if (!run || k < 1) { ser_set_error("ser_run_cross_chain: bad argument"); return SER_E_ARG; }
  if (run->cfg.store < SER_STORE_PI) { ser_set_error("ser_run_cross_chain: run has no pi sample store"); return SER_E_STATE; }
  if (run->acc_what || run->h_chain_ids) {
    ser_set_error("ser_run_cross_chain: needs a contiguous block of chains that stores all its samples (not a subset or accumulating run)");
    return SER_E_STATE;
  }
  if (set_device(run)) return SER_E_CUDA;
  int ranks = 1, rank = 0;
  if (comm && comm_ranks(comm, &ranks, &rank)) return SER_E_ARG;
  const int nl = run->cfg.n_chains, total = nl * ranks, N = run->N;
  if (run->cfg.chain_offset < rank * nl) {
    ser_set_error("ser_run_cross_chain: rank %d holds chain_offset %d; ranks hold consecutive blocks of %d chains", rank, run->cfg.chain_offset, nl);
    return SER_E_ARG;
  }
  if (run->cc_k != k || run->cc_total != total) { /* (re)size the step's device buffers */
    void *old[] = {run->d_e_all, run->d_info, run->d_chosen, run->d_counts};
    for (void *b : old) if (b) cudaFreeAsync(b, run->stream);
    run->d_e_all = nullptr; run->d_info = nullptr; run->d_chosen = nullptr; run->d_counts = nullptr;
    run->cc_k = 0;
    CUDA_TRY(POOL_ALLOC(&run->d_e_all, (size_t)total * sizeof(double)));
    CUDA_TRY(POOL_ALLOC(&run->d_info, 3 * sizeof(double)));
    CUDA_TRY(POOL_ALLOC(&run->d_chosen, (size_t)k * sizeof(int)));
    CUDA_TRY(POOL_ALLOC(&run->d_counts, (size_t)k * N * N * sizeof(int)));
    run->cc_k = k; run->cc_total = total;
  }
  run->cc_ranks = ranks; run->cc_rank = rank; run->cc_valid = 0;
  int rc = run_stats_to(run, one_dest(run->d_e_all), rank * nl); /* straight into this rank's slot of the gather buffer */
  if (rc) return rc;
  if (comm && (rc = comm_all_gather_e(comm, run->d_e_all, nl, run->stream))) return rc;
  mark_launch(run);
  ser_select_kernel<<<1, 1024, 0, run->stream>>>(run->d_e_all, total, k, run->d_chosen, run->d_info);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemsetAsync(run->d_counts, 0, (size_t)k * N * N * sizeof(int), run->stream));
  /* the selection numbers the chains by their index in the gathered array: this rank's chain 0 is rank * nl there */
  if ((rc = run_po_to(run, run->d_chosen, k, one_dest(run->d_counts), rank * nl))) return rc;
  if (comm && (rc = comm_all_reduce_counts(comm, run->d_counts, (size_t)k * N * N, run->stream))) return rc;
  run->cc_valid = 1;
  return SER_OK;
}

extern "C" int ser_run_cross_chain_result(ser_run *run, int32_t *chosen, int32_t *n_chosen, double *min_out, double *sigma_out,
                                          int32_t *counts)
{
  if (!run) return SER_E_ARG;
  if (!run->cc_valid) { ser_set_error("ser_run_cross_chain_result: call ser_run_cross_chain_async first"); return SER_E_STATE; }
  if (set_device(run)) return SER_E_CUDA;
  const int k = run->cc_k, N = run->N;
  double info[3] = {0, 0, 0};
  std::vector<int> ch(k, -1);
  CUDA_TRY(cudaMemcpyAsync(info, run->d_info, sizeof(info), cudaMemcpyDeviceToHost, run->stream));
  CUDA_TRY(cudaMemcpyAsync(ch.data(), run->d_chosen, (size_t)k * sizeof(int), cudaMemcpyDeviceToHost, run->stream));
  if (counts) CUDA_TRY(cudaMemcpyAsync(counts, run->d_counts, (size_t)k * N * N * sizeof(int), cudaMemcpyDeviceToHost, run->stream));
  CUDA_TRY(cudaStreamSynchronize(run->stream));
  const int base = run->cfg.chain_offset - run->cc_rank * run->cfg.n_chains; /* index in the gathered array -> GLOBAL id */
  if (chosen) for (int i = 0; i < k; i++) chosen[i] = ch[i] < 0 ? -1 : ch[i] + base;
  if (n_chosen) *n_chosen = (int)info[0];
  if (min_out) *min_out = info[1];
  if (sigma_out) *sigma_out = info[2];
  return SER_OK;
}

extern "C" int ser_run_cross_chain_buffers(ser_run *run, double **d_e_all, int32_t **d_chosen, double **d_info, int32_t **d_counts)
{
  if (!run || !run->cc_valid) { ser_set_error("ser_run_cross_chain_buffers: no cross-chain step enqueued"); return SER_E_STATE; }
  if (d_e_all) *d_e_all = run->d_e_all;
  if (d_chosen) *d_chosen = run->d_chosen;
  if (d_info) *d_info = run->d_info;
  if (d_counts) *d_counts = run->d_counts;
  return SER_OK;
}

/* out[0..2] = fp64 FMA TFLOP/s, shared-memory load GB/s, popc Gop/s; out[3..5] (ser_microbench_ex) = the kernel
 * times in ms they were derived from; work = blocks x threads x iters x {8 FMA x 2 flop, 8 x 16 B, 8 popc} */
extern "C" int ser_microbench_ex(int32_t device, double out[6])
{
  if (!out) return SER_E_ARG;
  CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  const int blocks = prop.multiProcessorCount * 2, threads = 1024, iters = 20000;
  void *buf = nullptr;
  CUDA_TRY(cudaMalloc(&buf, (size_t)blocks * threads * 8));
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
  float ms = 0.f;
  for (int rep = 0; rep < 2; rep++) { /* first pass warms up */
    CUDA_TRY(cudaEventRecord(e0));
    mb_fp64_kernel<<<blocks, threads>>>((double *)buf, iters);
    CUDA_TRY(cudaEventRecord(e1)); CUDA_TRY(cudaEventSynchronize(e1));
    CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
  }
  out[0] = (double)blocks * threads * iters * 8.0 * 2.0 / (ms * 1e-3) / 1e12; out[3] = ms;
  for (int rep = 0; rep < 2; rep++) {
    CUDA_TRY(cudaEventRecord(e0));
    mb_lds_kernel<<<blocks, threads>>>((unsigned *)buf, iters / 4);
    CUDA_TRY(cudaEventRecord(e1)); CUDA_TRY(cudaEventSynchronize(e1));
    CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
  }
  out[1] = (double)blocks * threads * (iters / 4) * 8.0 * 16.0 / (ms * 1e-3) / 1e9; out[4] = ms;
  for (int rep = 0; rep < 2; rep++) {
    CUDA_TRY(cudaEventRecord(e0));
    mb_popc_kernel<<<blocks, threads>>>((unsigned *)buf, iters);
    CUDA_TRY(cudaEventRecord(e1)); CUDA_TRY(cudaEventSynchronize(e1));
    CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
  }
  out[2] = (double)blocks * threads * iters * 8.0 / (ms * 1e-3) / 1e9; out[5] = ms;
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(buf);
  return SER_OK;
}

extern "C" int ser_microbench(int32_t device, double out[3])
{
  double all[6];
  if (!out) return SER_E_ARG;
  const int rc = ser_microbench_ex(device, all);
  if (rc) return rc;
  out[0] = all[0]; out[1] = all[1]; out[2] = all[2];
  return SER_OK;
}

#include "ser_multi.cuh"
#include "ser_ckpt.cuh"
