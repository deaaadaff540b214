/* ser_device_common.cuh -- kernel parameters, the shared-memory carve-up, block helpers and the init kernel.
 * Part of the single translation unit ser_kernels.cu (included there, in this order). */

/* phase timing of the sweep kernels (debug builds: NVCC_EXTRA=-DSER_PHASE_TIMING): thread 0 of every
 * CTA adds the cycles between marks; ser_debug_phase_cycles() reads and clears the totals */
#ifdef SER_PHASE_TIMING
__device__ unsigned long long ser_phase_cycles[24];
#define PHASE_T0() long long ph_t = clock64()
#define PHASE_MARK(i) do { if (threadIdx.x == 0) { const long long ph_n = clock64(); atomicAdd(&ser_phase_cycles[i], (unsigned long long)(ph_n - ph_t)); ph_t = ph_n; } } while (0)
extern "C" int ser_debug_phase_cycles(unsigned long long out[24])
{
  unsigned long long zero[24] = {0};
  if (cudaDeviceSynchronize() != cudaSuccess || cudaMemcpyFromSymbol(out, ser_phase_cycles, sizeof(zero)) != cudaSuccess) return -1;
  return cudaMemcpyToSymbol(ser_phase_cycles, zero, sizeof(zero)) == cudaSuccess ? 0 : -1;
}
#else
#define PHASE_T0() do { } while (0)
#define PHASE_MARK(i) do { } while (0)
#endif

/* The large-shape kernel's columns live in a global scratch slot per CTA; 148 slots of bit columns + per-word prefix counts are
 * the size of the L2 (1024 x 4096: 0.54 + 0.28 MB each).  One prefix count per 2^SER_BIG_G words (ser_pre_at, ser_chain_core.h)
 * shrinks the table by that factor; the words between an entry and the word asked for are counted on the fly.  Measured with
 * -DSER_BIG_G=2 (parity green): DRAM traffic 2.47 -> 1.18 GB per 2 960 chain-sweeps, but 13 % more instructions and
 * instruction-cache misses: 242 -> 197 k sweeps/s (-DSER_BIG_G=1: 201 k).  The default stays one count per word. */
#ifndef SER_BIG_G
#define SER_BIG_G 0
#endif

/* ------------------------------------------------------------------ per-chain global state */
struct __align__(16) ChainScalars { /* a multiple of 16 bytes: loaded / stored as int4 words */
  double c, cc, d, dd; /* log P(false 1), log(1-e^c), log P(false 0), log(1-e^d) */
  double loglik;
  double sum_negll, sum_ec, sum_ed; /* compute_exp_data, mcmc.c:53-58 */
  long long cursor;                 /* replay: tape slots consumed */
  long long counters[8];            /* c, d, ab changed, pi1, pi2(0), pi2(swap), pi3, sweeps */
  int t0a, f0a, t1a, f1a;
  unsigned int sweep; /* free-running: sweep index = Philox counter word */
  int n_samples;
  int flags; /* bit0 tape exhausted, bits 1-4 consistency failures (ser_check_kernel), bit5 bit columns stored in gVc */
  int pad;
  long long pad2;
};
static_assert(sizeof(ChainScalars) % 16 == 0, "ChainScalars is moved as int4 words");
#define SER_FLAG_COLUMNS 32

struct KParams {
  int N, M, W, C, nh, Mw, Npad, Mpad;
  const uint32_t *Xs;  /* [N][Mw] site-major bits */
  const uint8_t *hard; /* [N] file order */
  const int *ones;     /* [M] ones per column */
  const uint16_t *order;    /* [M] column -> taxon (columns are sorted by ones, descending) */
  const int *off;           /* [M+1] first item of each column; a column has ones+1 items */
  const uint32_t *item_col; /* [I] item -> (column << 16) | index of the item inside its column */
  const uint16_t *col_sites; /* [ones_total] the sites (file order) holding a one, per sorted column; column c starts at off[c] - c */
  const uint32_t *hbits;    /* [M] bit k = the column has a one at the k-th hard site in file order (first 32 hard sites) */
  int I;                    /* ones_total + M */
  /* large-shape path (ser_sweep_kernel_big): per-CTA-slot scratch in global memory */
  int Cs;                   /* column stride of the scratch bit matrix (>= M+1) */
  uint32_t *gV;             /* [slot][W][Cs] */
  uint16_t *gpre;           /* [slot][(W >> SER_BIG_G) + 1][Cs]: one prefix count per 2^SER_BIG_G words */
  const int *bgrp;          /* large-shape column groups: [g] = {first column, first item}, big_ng + 1 entries */
  int big_ng, big_icap, big_gcap;
  /* warp-batch Gibbs phase (ser_sweep_kernel_big<.., WB = true>): a batch = consecutive columns one warp serves on its own */
  const int4 *bbat;         /* [big_nb] = {first column, columns | lane shift << 16, first item, last item + 1} */
  int big_nb, big_wcap;     /* batches; items per warp slice of the item buffers */
  int n_chains;
  uint16_t *ab;        /* [chain][2][Mpad] */
  uint16_t *rpi;       /* [chain][Npad] */
  ChainScalars *scal;  /* [chain] */
  int mode, chain_offset;
  const int *chain_ids;     /* [n_chains] global id of each local chain (ser_run_create_chains), else nullptr: chain_offset + chain */
  unsigned int seed;
  const double *tape;
  const unsigned long long *tape_off;
  int n_calls, sweeps_per_call;
  int burn_calls;           /* calls [0, burn_calls) of a launch are burn-in, the rest emit a thinned sample each */
  /* persistent work-queue grid (ser_sweep_kernel): items = chunks of chunk_calls calls of one chain */
  unsigned int n_items, chunk_base; /* items of this launch; done[chain] before the launch */
  int chunk_calls;
  uint32_t *gVc;            /* [chain][W][C] bit columns carried between work items */
  unsigned int *queue;      /* next item */
  unsigned int *done;       /* [chain] items completed since init */
  int store, max_samples;
  int sample_base;          /* samples taken before the store's row 0: 0, or on an accumulating run those already summarised */
  uint16_t *samp_a, *samp_b, *samp_pi;
  double *samp_cdl;
  double c0, cc0, d0, dd0, eps;
  long long ones_total;
  /* per-taxon c, d (manycd = 1, mcmc.c:777-785, :807-815) */
  int manycd;
  double *cd4;         /* [chain][4][Mpad]: c, log(1-e^c), d, log(1-e^d) per column */
  double *samp_cd_all; /* [chain][sample][2][M]: c, d per taxon (SER_STORE_FULL) */
  int col0;            /* the sorted column that holds taxon 0 (its c, d are what compute_exp_data reads) */
  /* the item weights of a Gibbs step are evaluated group by group of columns through a buffer of
   * Ival doubles: a smaller buffer = more resident chains per SM */
  int n_groups, Ival;
  int grp_c[SER_MAX_GROUPS + 1], grp_e[SER_MAX_GROUPS + 1];
  /* units of the Gibbs phase: heavy columns are served by 2, 4, .. 32 adjacent lanes (ser_sweep_kernel.cuh) */
  const uint2 *unit_tab; /* [n_units] = {column | sub << 16 | lsh << 24, first item of the column} */
  int n_units;
  int grp_u[SER_MAX_GROUPS + 1]; /* units of column group g = [grp_u[g], grp_u[g+1]) */
};

/* the global chain id that keys local chain `chain`'s Philox stream */
__device__ __forceinline__ unsigned int global_chain(const KParams &p, int chain)
{
  return (unsigned int)(p.chain_ids ? p.chain_ids[chain] : p.chain_offset + chain);
}

/* ------------------------------------------------------------------ shared-memory carve-up */
struct Smem {
  double *draws_pi; /* SER_PI_DRAWS */
  double *logdraw;  /* SER_PI_DRAWS: log of each staged draw (only read where a draw is a U+) */
  double *draws_cd; /* 8 */
  double *terms;    /* C */
  double *H;        /* N + 2: geometric partial sums of the current sweep (ser_h_entry) */
  uint32_t *V;      /* W*C */
  int *red;         /* 2 * SER_MAX_WARPS * 4 */
  double *val;      /* I+1: item weights of the running Gibbs step */
  double *lmax;     /* C: per-column maximum log-weight of the running step */
  uint16_t *pos;    /* I+1: ascending positions of the ones of every column (postings) */
  uint16_t *st4;    /* 4*C: per-column step geometry: cur, bound, ocur, kb */
  uint16_t *ones16; /* C: ones per column (static; keeps the dense item loop free of dependent global loads) */
  uint16_t *pre;    /* (W+1)*C: pre[w][col] = ones of the column in words < w */
  uint16_t *hp;     /* N+1: hard positions, ascending */
  double *wcol;     /* manycd only: 4*C per-column weights A, g, 1/g, 1/(1-e^-g) for the dense item phase */
  double *redd;     /* manycd only: 2*32 doubles of reduction scratch */
  uint16_t *rpi, *tmp16, *perm16; /* N each; tmp16 / perm16 (staging of an accepted move) share their bytes with ncache */
  uint16_t *pick16; /* C: the item the column's uniform fell into (Gibbs step) */
  uint16_t *ncache; /* Ival + 1 run lengths of the running group's items (written by the maximum pass, read by the dense pass) */
  uint16_t *hrank, *nhpos; /* N+2 each: hard positions before p; position of the r-th non-hard site (SerHard's tables) */
};

__host__ __device__ inline size_t smem_layout(Smem *s, unsigned char *base, int N, int W, int C, int I, int manycd = 0, int Ival = -1)
{
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 15) & ~(size_t)15; return o; };
  size_t o_ld = take(sizeof(double) * SER_PI_DRAWS);
  size_t o_dp = take(sizeof(double) * SER_PI_DRAWS), o_dc = take(sizeof(double) * 8), o_t = take(sizeof(double) * C);
  size_t o_H = take(sizeof(double) * (N + 2 < SER_HCAP ? N + 2 : SER_HCAP));
  /* the run-length cache of the Gibbs phase and the two staging arrays of an accepted site move are never live together */
  const size_t nc_bytes = sizeof(uint16_t) * ((Ival < 0 ? I : Ival) + 1), st_bytes = 2 * ((sizeof(uint16_t) * N + 15) & ~(size_t)15);
  size_t o_nc = take(nc_bytes > st_bytes ? nc_bytes : st_bytes);
  size_t o_val = take(sizeof(double) * ((Ival < 0 ? I : Ival) + 1)), o_lm = take(sizeof(double) * C);
  size_t o_wc = take(manycd ? sizeof(double) * 4 * C : 0), o_rd = take(manycd ? sizeof(double) * 2 * SER_MAX_WARPS : 0);
  size_t o_pos = take(sizeof(uint16_t) * (I + 1)), o_st = take(sizeof(uint16_t) * 4 * C), o_on = take(sizeof(uint16_t) * C);
  size_t o_v = take(sizeof(uint32_t) * (size_t)W * C), o_r = take(sizeof(int) * 2 * SER_MAX_WARPS * 4);
  size_t o_h = take(sizeof(uint16_t) * (size_t)(W + 1) * C), o_hp = take(sizeof(uint16_t) * (N + 1));
  size_t o_p = take(sizeof(uint16_t) * N), o_q = o_nc, o_m = o_nc + ((sizeof(uint16_t) * N + 15) & ~(size_t)15);
  size_t o_hr = take(sizeof(uint16_t) * (N + 2)), o_nh = take(sizeof(uint16_t) * (N + 2)), o_pk = take(sizeof(uint16_t) * C);
  if (s) {
    s->pick16 = (uint16_t *)(base + o_pk);
    s->hrank = (uint16_t *)(base + o_hr); s->nhpos = (uint16_t *)(base + o_nh);
    s->logdraw = (double *)(base + o_ld);
    s->draws_pi = (double *)(base + o_dp); s->draws_cd = (double *)(base + o_dc); s->terms = (double *)(base + o_t);
    s->H = (double *)(base + o_H); s->ncache = (uint16_t *)(base + o_nc);
    s->val = (double *)(base + o_val); s->lmax = (double *)(base + o_lm);
    s->wcol = (double *)(base + o_wc); s->redd = (double *)(base + o_rd);
    s->pos = (uint16_t *)(base + o_pos); s->st4 = (uint16_t *)(base + o_st); s->ones16 = (uint16_t *)(base + o_on);
    s->V = (uint32_t *)(base + o_v); s->red = (int *)(base + o_r); s->pre = (uint16_t *)(base + o_h); s->hp = (uint16_t *)(base + o_hp);
    s->rpi = (uint16_t *)(base + o_p); s->tmp16 = (uint16_t *)(base + o_q); s->perm16 = (uint16_t *)(base + o_m);
  }
  return off;
}

/* ------------------------------------------------------------------ block helpers */
/* sum of three ints over the CTA; every thread gets the totals.  One __syncthreads; `buf`
 * alternates between calls so a warp that runs ahead never overwrites live partials. */
__device__ __forceinline__ void block_sum3(int v0, int v1, int v2, int *red, int &buf, int *o0, int *o1, int *o2)
{
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
  v0 = __reduce_add_sync(0xffffffffu, v0);
  v1 = __reduce_add_sync(0xffffffffu, v1);
  v2 = __reduce_add_sync(0xffffffffu, v2);
  int *r = red + buf * (SER_MAX_WARPS * 4);
  if (lane == 0) { r[warp * 4 + 0] = v0; r[warp * 4 + 1] = v1; r[warp * 4 + 2] = v2; }
  __syncthreads();
  /* second level: lane w picks up warp w's partials, one more REDUX per value */
  int s0 = 0, s1 = 0, s2 = 0;
  if (lane < nwarp) { s0 = r[lane * 4 + 0]; s1 = r[lane * 4 + 1]; s2 = r[lane * 4 + 2]; }
  s0 = __reduce_add_sync(0xffffffffu, s0);
  s1 = __reduce_add_sync(0xffffffffu, s1);
  s2 = __reduce_add_sync(0xffffffffu, s2);
  buf ^= 1;
  *o0 = s0; *o1 = s1; *o2 = s2;
}

/* position-ordered columns from the site-major data and rpi; column M = hard mask */
__device__ void build_columns(const KParams &p, const Smem &sm)
{
  const int tid = threadIdx.x, C = p.C;
  const int mw = tid >> 5, mb = tid & 31;
  for (int w = 0; w < p.W; w++) {
    uint32_t word = 0;
    const int pend = min(32 * w + 32, p.N);
    if (tid < p.M) {
      for (int pos = 32 * w; pos < pend; pos++)
        word |= ((p.Xs[(size_t)sm.rpi[pos] * p.Mw + mw] >> mb) & 1u) << (pos & 31);
    } else if (tid == p.M) {
      for (int pos = 32 * w; pos < pend; pos++) word |= (uint32_t)(p.hard[sm.rpi[pos]] != 0) << (pos & 31);
    }
    sm.V[w * C + tid] = word;
  }
  ser_col_build_pre(sm.V + tid, sm.pre + tid, C, p.W);
}

/* The hard-site tables from the hard-mask column, by all threads of the CTA (the column must be complete: barrier
 * before; the tables are complete after the next barrier): hrank[q] = hard positions < q, hp[k] = position of the
 * k-th hard site, nhpos[r] = position of the r-th non-hard site. */
__device__ __forceinline__ void rebuild_hard(const KParams &p, const Smem &sm)
{
  const uint32_t *hcol = sm.V + p.M;
  const uint16_t *hpre = sm.pre + p.M;
  for (int q = threadIdx.x; q <= p.N; q += blockDim.x) {
    const int r = ser_rank1(hcol, hpre, p.C, q);
    sm.hrank[q] = (uint16_t)r;
    if (q < p.N) {
      if ((hcol[(q >> 5) * p.C] >> (q & 31)) & 1u) sm.hp[r] = (uint16_t)q;
      else sm.nhpos[q - r] = (uint16_t)q;
    }
  }
}

__device__ __forceinline__ void set_weights(SerWeights &wt, double c, double cc, double d, double dd)
{
  ser_set_weights(&wt, c, cc, d, dd);
}

/* totals and log-likelihood from the block-reduced alive-ones / lifespan sums (mcmc.c:977-986) */
__device__ __forceinline__ void totals_from(const KParams &p, const SerWeights &wt, int T1, int LEN, int *t0a, int *f0a,
                                            int *t1a, int *f1a, double *loglik)
{
  const int f1 = (int)p.ones_total - T1, f0 = LEN - T1, t0 = p.N * p.M - LEN - f1;
  *t1a = T1; *f1a = f1; *f0a = f0; *t0a = t0;
  *loglik = SER_ADD(SER_ADD(SER_ADD(SER_MUL((double)t0, wt.cc), SER_MUL((double)f0, wt.d)), SER_MUL((double)T1, wt.dd)),
                    SER_MUL((double)f1, wt.c));
}

/* ------------------------------------------------------------------ V-free helpers
 * The init / export / check kernels do not need the bit columns: a thread walks its taxa's cells in
 * position order straight from the site-major matrix.  They work for every shape. */
__device__ __forceinline__ int cell(const KParams &p, const uint16_t *rpi, int pos, int c)
{
  return (p.Xs[(size_t)rpi[pos] * p.Mw + (c >> 5)] >> (c & 31)) & 1u;
}
__device__ int taxon_count(const KParams &p, const uint16_t *rpi, int c, int lo, int hi)
{
  int n = 0;
  for (int pos = lo; pos < hi; pos++) n += cell(p, rpi, pos, c);
  return n;
}
/* mcmc_initab, mcmc.c:440-474 */
__device__ void taxon_init_ab(const KParams &p, const uint16_t *rpi, int c, int *a, int *b)
{
  int first = -1, last = -1;
  for (int pos = 0; pos < p.N; pos++)
    if (cell(p, rpi, pos, c)) { if (first < 0) first = pos; last = pos; }
  if (first < 0) { *a = 0; *b = p.N; } else { *a = first; *b = last + 1; }
}

struct AuxSmem { /* init / export / check kernels */
  int *red;
  uint16_t *rpi, *tmp16;
};
__host__ __device__ inline size_t aux_layout(AuxSmem *s, unsigned char *base, int N)
{
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 15) & ~(size_t)15; return o; };
  size_t o_r = take(sizeof(int) * 2 * SER_MAX_WARPS * 4), o_p = take(sizeof(uint16_t) * N), o_t = take(sizeof(uint16_t) * N);
  if (s) { s->red = (int *)(base + o_r); s->rpi = (uint16_t *)(base + o_p); s->tmp16 = (uint16_t *)(base + o_t); }
  return off;
}

/* ------------------------------------------------------------------ init kernel */
/* mcmc_readmodel's initial state + mcmc_randomize (mcmc.c:405-433, :477-578) */
__global__ void ser_init_kernel(KParams p)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  AuxSmem sm;
  const size_t used = aux_layout(&sm, smem_raw, p.N);
  /* behind the common layout: 2N staged draws, pi / rest / chosen as u16 */
  double *stage = (double *)(smem_raw + used);
  uint16_t *pi16 = (uint16_t *)(stage + 2 * p.N);
  uint16_t *rest16 = pi16 + p.N, *chosen16 = rest16 + p.N;

  const int chain = blockIdx.x, tid = threadIdx.x, N = p.N, M = p.M, C = blockDim.x, nh = p.nh;
  const double *tape = nullptr;
  long long tape_len = 0;
  if (p.mode == SER_MODE_REPLAY) {
    tape = p.tape + p.tape_off[chain];
    tape_len = (long long)(p.tape_off[chain + 1] - p.tape_off[chain]);
  }
  /* the global id is formed where it is used: held across the kernel it costs 8 registers, a resident block per SM at 320 threads */
  for (int t = tid; t < 2 * N; t += C) {
    if (p.mode == SER_MODE_REPLAY) stage[t] = (t < tape_len) ? tape[t] : 0.0;
    else stage[t] = ser_stream_uniform(p.seed, global_chain(p, chain), SER_SWEEP_INIT, SER_BLK_INIT, (uint32_t)t);
  }
  for (int n = tid; n < N; n += C) sm.rpi[n] = (uint16_t)n;
  __syncthreads();

  uint16_t *ab = p.ab + (size_t)chain * 2 * p.Mpad;
  __shared__ int s_used;
  if (tid == 0) {
    int used_draws = 0;
    for (int n = 0; n < N; n++) pi16[n] = (uint16_t)n;
    if (nh == 0) {
      for (int i = N - 1; i > 0; i--) {
        const int j = ser_draw_int(stage[used_draws++], i + 1);
        const uint16_t t = pi16[i]; pi16[i] = pi16[j]; pi16[j] = t;
      }
    } else if (nh < N) {
      int j = 0;
      for (int i = 0; i < N && j < nh; i++)
        if (SER_MUL((double)(N - i), stage[used_draws++]) < (double)(nh - j)) chosen16[j++] = (uint16_t)i;
      int k = 0;
      j = 0;
      for (int i = 0; i < N; i++) {
        if (j < nh && i == chosen16[j]) j++;
        else rest16[k++] = (uint16_t)i;
      }
      for (int i = N - nh - 1; i > 0; i--) {
        const int r = ser_draw_int(stage[used_draws++], i + 1);
        const uint16_t t = rest16[i]; rest16[i] = rest16[r]; rest16[r] = t;
      }
      j = k = 0;
      for (int i = 0; i < N; i++) pi16[i] = p.hard[i] ? chosen16[j++] : rest16[k++];
    }
    s_used = used_draws;
  }
  __syncthreads();
  for (int n = tid; n < N; n += C) sm.rpi[pi16[n]] = (uint16_t)n;
  __syncthreads();

  SerWeights wt;
  wt.eps = p.eps;
  set_weights(wt, p.c0, p.cc0, p.d0, p.dd0);
  /* mcmc_initab (mcmc.c:440-474) + the alive ones of mcmc_count01 from the column's static site list (the sites that hold a
   * one, in file order): a = first, b = last + 1 position of a one, so every one is alive.  nh == 0: the identity-order
   * a, b are kept although pi was shuffled (mcmc.c:486-494) -- then the alive ones have to be counted. */
  int t1 = 0, len = 0;
  for (int c = tid; c < M; c += C) {
    const uint16_t *cs = p.col_sites + (p.off[c] - c);
    const int K = p.ones[c];
    int a = 0, b = N, t1c = 0;
    if (nh != 0) {
      int mn = N, mx = -1;
      for (int k = 0; k < K; k++) { const int q = pi16[cs[k]]; mn = min(mn, q); mx = max(mx, q); }
      if (K) { a = mn; b = mx + 1; }
      t1c = K;
    } else {
      if (K) { a = cs[0]; b = cs[K - 1] + 1; }
      for (int k = 0; k < K; k++) { const int q = pi16[cs[k]]; t1c += (a <= q && q < b); }
    }
    ab[c] = (uint16_t)a; ab[p.Mpad + c] = (uint16_t)b;
    t1 += t1c;
    len += b - a;
  }
  int buf = 0, T1, LEN, dummy;
  block_sum3(t1, len, 0, sm.red, buf, &T1, &LEN, &dummy);
  int t0a, f0a, t1a, f1a;
  double loglik;
  totals_from(p, wt, T1, LEN, &t0a, &f0a, &t1a, &f1a, &loglik);

  for (int n = tid; n < N; n += C) p.rpi[(size_t)chain * p.Npad + n] = sm.rpi[n];
  if (p.manycd)
    for (int c = tid; c < M; c += C) {
      double *cd = p.cd4 + (size_t)chain * 4 * p.Mpad + c;
      cd[0] = p.c0; cd[p.Mpad] = p.cc0; cd[2 * p.Mpad] = p.d0; cd[3 * p.Mpad] = p.dd0;
    }
  if (tid == 0) {
    ChainScalars sc;
    memset(&sc, 0, sizeof(sc));
    sc.c = p.c0; sc.cc = p.cc0; sc.d = p.d0; sc.dd = p.dd0;
    sc.loglik = loglik;
    sc.t0a = t0a; sc.f0a = f0a; sc.t1a = t1a; sc.f1a = f1a;
    sc.cursor = s_used;
    sc.flags = (p.mode == SER_MODE_REPLAY && s_used > tape_len) ? 1 : 0;
    p.scal[chain] = sc;
  }
}
