/* ser_sweep_kernel_cluster.cuh -- the large-shape sweep kernel on thread-block clusters: one chain per cluster of R CTAs,
 * the chain's bit columns resident in the cluster's shared memory.
 * Part of the single translation unit ser_kernels.cu (included there, in this order).
 *
 * Why: for 1024 sites x 4096 taxa the position-ordered bit columns (0.54 MB) and their prefix tables (0.28 MB) do not fit one
 * SM.  ser_sweep_kernel_big keeps them in a global scratch slot per CTA; 148 slots are the size of the L2, so every sweep
 * re-streams them from HBM (1.35 MB of DRAM traffic per chain-sweep against 1.8 KB algorithmic).  Here the columns are
 * SHARDED over the R CTAs of a cluster (column gc belongs to rank gc % R, so every rank holds the same mix of heavy and light
 * columns) and stay in shared memory for the life of a chain: nothing but the draw tape and the thinned samples touches
 * HBM inside a sweep.  Everything per-column -- the Gibbs step, the proposal deltas, the column rewrites of an accepted
 * move -- is local to the owning CTA.  What is shared by all taxa is replicated in every CTA and updated redundantly (site
 * order, hard-site mask and tables, c / d, the staged draws, the decisions).  The only exchange is the sum of the integer
 * deltas of a proposal (and of the Gibbs totals): each CTA stores its three partial sums into every CTA's shared memory
 * (DSMEM) and one cluster barrier publishes them -- 17 exchanges of 12 bytes per sweep.  The taxon-order float sums the
 * reference's bits require (saved log-likelihood, degenerate proposals) gather their terms in rank 0's shared memory.
 *
 * Reference: mcmc_sample and its sub-samplers, C_Implementation/mcmc.c:214-258, :751-996, :1127-1682 (as ser_sweep_kernel).
 */
#include <cooperative_groups.h>
namespace cg = cooperative_groups;

#define SER_CL_MAXR 8
#define SER_CL_HCAP 288 /* entries of the geometric-sum table: hmax <= -LOGEPSILON / g_min + 3 = 277 (g >= log .9 - log .8) */

struct ClSmem {
  double *draws_pi, *logdraw, *draws_cd, *H;
  double *lmax, *dsl; /* gcap: per column of the running group: maximum log-weight; target minus the weight before the picked item */
  double *xdbl;       /* 2: exact sums broadcast by rank 0 */
  double *val;        /* icap: item log-weights / weights / cumulative weights of the running group; TERMS outside the Gibbs phase */
  int *red, *xint;    /* block reduction scratch; [2][SER_CL_MAXR][4] partial sums of every rank (written through DSMEM) */
  int *goff;          /* gcap: first item of each column of the running group relative to the group's first item */
  uint16_t *a16, *b16;                  /* Mc: a, b of the local columns */
  uint16_t *hp, *rpi, *tmp16, *perm16;  /* replicated: hard positions, site order, scratch */
  uint16_t *hrank, *nhpos;              /* replicated: SerHard's tables */
  uint16_t *st4, *gones, *pick16;       /* 4 gcap, gcap, gcap */
  uint32_t *hb32;                       /* Mc: hard-site bits of the local columns */
  uint32_t *V;                          /* W x Cs: local columns (+ the hard mask at local column Mc) in position order */
  uint16_t *pre;                        /* (W+1) x Cs */
  uint16_t *pos;                        /* icap: postings of the running group's columns */
};

__host__ __device__ inline size_t cl_layout(ClSmem *s, unsigned char *base, int N, int W, int Mc, int icap, int gcap)
{
  const int Cs = Mc + 1, hcap = (N + 2 < SER_CL_HCAP) ? N + 2 : SER_CL_HCAP;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 15) & ~(size_t)15; return o; };
  size_t o_dp = take(8 * SER_PI_DRAWS), o_ld = take(8 * SER_PI_DRAWS), o_dc = take(8 * 8), o_H = take(8 * (size_t)hcap);
  size_t o_lm = take(8 * (size_t)gcap), o_ds = take(8 * (size_t)gcap), o_xd = take(8 * 2), o_val = take(8 * (size_t)icap);
  size_t o_r = take(sizeof(int) * 2 * SER_MAX_WARPS * 4), o_xi = take(sizeof(int) * 2 * SER_CL_MAXR * 4), o_go = take(4 * (size_t)gcap);
  size_t o_a = take(2 * (size_t)Mc), o_b = take(2 * (size_t)Mc), o_hp = take(2 * (size_t)(N + 1));
  size_t o_p = take(2 * (size_t)N), o_q = take(2 * (size_t)N), o_m = take(2 * (size_t)N);
  size_t o_hr = take(2 * (size_t)(N + 2)), o_nh = take(2 * (size_t)(N + 2));
  size_t o_st = take(2 * 4 * (size_t)gcap), o_gn = take(2 * (size_t)gcap), o_pk = take(2 * (size_t)gcap), o_hb = take(4 * (size_t)Mc);
  size_t o_v = take(4 * (size_t)W * Cs), o_pre = take(2 * (size_t)(W + 1) * Cs), o_pos = take(2 * (size_t)icap);
  if (s) {
    s->draws_pi = (double *)(base + o_dp); s->logdraw = (double *)(base + o_ld); s->draws_cd = (double *)(base + o_dc); s->H = (double *)(base + o_H);
    s->lmax = (double *)(base + o_lm); s->dsl = (double *)(base + o_ds); s->xdbl = (double *)(base + o_xd); s->val = (double *)(base + o_val);
    s->red = (int *)(base + o_r); s->xint = (int *)(base + o_xi); s->goff = (int *)(base + o_go);
    s->a16 = (uint16_t *)(base + o_a); s->b16 = (uint16_t *)(base + o_b); s->hp = (uint16_t *)(base + o_hp);
    s->rpi = (uint16_t *)(base + o_p); s->tmp16 = (uint16_t *)(base + o_q); s->perm16 = (uint16_t *)(base + o_m);
    s->hrank = (uint16_t *)(base + o_hr); s->nhpos = (uint16_t *)(base + o_nh);
    s->st4 = (uint16_t *)(base + o_st); s->gones = (uint16_t *)(base + o_gn); s->pick16 = (uint16_t *)(base + o_pk); s->hb32 = (uint32_t *)(base + o_hb);
    s->V = (uint32_t *)(base + o_v); s->pre = (uint16_t *)(base + o_pre); s->pos = (uint16_t *)(base + o_pos);
  }
  return off;
}

/* sum of three ints over ALL threads of the cluster.  Block level as block_sum3; then every CTA stores its three sums into
 * slot [buf][rank] of every CTA (DSMEM) and one cluster barrier makes them visible.  `buf` alternates: a CTA that runs ahead
 * writes the other half, and cannot come back to this half before everybody has passed the next barrier. */
__device__ __forceinline__ void cluster_sum3(cg::cluster_group &cluster, const ClSmem &sm, int R, int rank, int v0, int v1, int v2, int &buf,
                                             int *o0, int *o1, int *o2)
{
  int rb = 0, s0, s1, s2;
  block_sum3(v0, v1, v2, sm.red, rb, &s0, &s1, &s2);
  if ((int)threadIdx.x < R) {
    int *dst = cluster.map_shared_rank(sm.xint, threadIdx.x) + (buf * SER_CL_MAXR + rank) * 4;
    dst[0] = s0; dst[1] = s1; dst[2] = s2;
  }
  cluster.sync();
  int t0 = 0, t1 = 0, t2 = 0;
  for (int q = 0; q < R; q++) {
    const int *src = sm.xint + (buf * SER_CL_MAXR + q) * 4;
    t0 += src[0]; t1 += src[1]; t2 += src[2];
  }
  buf ^= 1;
  *o0 = t0; *o1 = t1; *o2 = t2;
}

/* The M per-taxon terms were stored into rank 0's TERMS (= its val buffer) by their owners: rank 0 adds them in taxon order
 * (the reference's own order of additions, mcmc.c:625-648 / :1214) and hands the sum to every CTA. */
__device__ __forceinline__ double cluster_sequential_sum(cg::cluster_group &cluster, const ClSmem &sm, int R, int rank, int M)
{
  cluster.sync(); /* all terms have arrived */
  if (rank == 0 && threadIdx.x < 32) { /* one warp walks the dependent chain (see sequential_term_sum) */
    double acc = 0.0;
    for (int m = 0; m < M; m++) acc = SER_ADD(acc, sm.val[m]);
    if (threadIdx.x == 0)
      for (int q = 0; q < R; q++) cluster.map_shared_rank(sm.xdbl, q)[0] = acc;
  }
  cluster.sync();
  return sm.xdbl[0];
}

/* MH tail (mh_decide / mh_decide_big) over the cluster: `redo(lc, &dt0, &dt1)` re-evaluates a local column's deltas */
template <typename Redo>
__device__ __forceinline__ bool mh_decide_cl(cg::cluster_group &cluster, const KParams &p, const ClSmem &sm, const SerWeights &wt, PropState &ps,
                                             int R, int rank, int nloc, int dt0, int dt1, int nz, bool exact, int *D0, int *D1,
                                             double *delta_out, Redo redo)
{
  int NZ;
  cluster_sum3(cluster, sm, R, rank, dt0, dt1, nz, ps.buf, D0, D1, &NZ);
  auto reference_sum = [&]() {
    double *T0 = cluster.map_shared_rank(sm.val, 0);
    for (int lc = threadIdx.x; lc < nloc; lc += blockDim.x) {
      int x0, x1;
      redo(lc, &x0, &x1);
      T0[p.order[lc * R + rank]] = ser_term(wt, x0, x1);
    }
    return cluster_sequential_sum(cluster, sm, R, rank, p.M);
  };
  double delta;
  bool seq = false;
  if (*D0 == 0 && *D1 == 0) {
    delta = 0.0;
    if (NZ) { delta = reference_sum(); seq = true; }
  } else {
    delta = ser_term(wt, *D0, *D1);
  }
  bool accept = delta >= 0.0;
  if (!accept) accept = delta > sm.logdraw[ps.k++];
  if (accept && exact && !seq && NZ) delta = reference_sum();
  *delta_out = delta;
  return accept;
}

/* hard-site tables of this CTA's replica (as rebuild_hard) */
__device__ __forceinline__ void cl_rebuild_hard(const ClSmem &sm, int N, int Mc, int Cs)
{
  const uint32_t *hcol = sm.V + Mc;
  const uint16_t *hpre = sm.pre + Mc;
  for (int q = threadIdx.x; q <= N; q += blockDim.x) {
    const int r = ser_rank1(hcol, hpre, Cs, q);
    sm.hrank[q] = (uint16_t)r;
    if (q < N) {
      if ((hcol[(q >> 5) * Cs] >> (q & 31)) & 1u) sm.hp[r] = (uint16_t)q;
      else sm.nhpos[q - r] = (uint16_t)q;
    }
  }
}

__global__ void __launch_bounds__(1024, 1) ser_sweep_kernel_cl(KParams p)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ unsigned int s_gchain;
  cg::cluster_group cluster = cg::this_cluster();
  const int R = p.cl_R, rank = (int)cluster.block_rank(), n_clusters = (int)gridDim.x / R, cid = (int)blockIdx.x / R;
  const int tid = threadIdx.x, N = p.N, M = p.M, C = blockDim.x, W = p.W, Mc = p.cl_Mc, Cs = Mc + 1;
  const int nloc = (M - rank + R - 1) / R; /* local column lc <-> sorted column lc * R + rank */
  ClSmem sm;
  cl_layout(&sm, smem_raw, N, W, Mc, p.cl_icap, p.cl_gcap);
  uint32_t *V = sm.V;
  uint16_t *PRE = sm.pre;
  double *TERMS0 = cluster.map_shared_rank(sm.val, 0); /* rank 0's term buffer (idle outside the Gibbs phase; icap >= M) */
  const int *grp = p.cl_grp + 2 * p.cl_grp_base[rank];
  const int ng = p.cl_grp_base[rank + 1] - p.cl_grp_base[rank] - 1;
  const uint32_t *items = p.cl_item + p.cl_item_base[rank];

  for (int lc = tid; lc < nloc; lc += C) sm.hb32[lc] = p.hbits[lc * R + rank];

  for (int chain = cid; chain < p.n_chains; chain += n_clusters) {
    const unsigned int &gchain = s_gchain; /* in shared memory, like ser_sweep_kernel's */
    __syncthreads(); /* the previous chain is done with this CTA's shared memory */
    if (threadIdx.x == 0) s_gchain = global_chain(p, chain); /* visible after the next barrier */
    ChainScalars sc = p.scal[chain];
    for (int n = tid; n < N; n += C) sm.rpi[n] = p.rpi[(size_t)chain * p.Npad + n];
    for (int lc = tid; lc < nloc; lc += C) {
      sm.a16[lc] = p.ab[(size_t)chain * 2 * p.Mpad + lc * R + rank];
      sm.b16[lc] = p.ab[(size_t)chain * 2 * p.Mpad + p.Mpad + lc * R + rank];
    }
    __syncthreads();
    /* position-ordered local columns + prefix tables; local column Mc = this CTA's copy of the hard mask */
    for (int lc = tid; lc <= Mc; lc += C) {
      const int gc = lc * R + rank;
      for (int w = 0; w < W; w++) {
        uint32_t word = 0;
        const int pend = min(32 * w + 32, N);
        if (lc < nloc) { for (int pos = 32 * w; pos < pend; pos++) word |= (uint32_t)cell(p, sm.rpi, pos, gc) << (pos & 31); }
        else if (lc == Mc) { for (int pos = 32 * w; pos < pend; pos++) word |= (uint32_t)(p.hard[sm.rpi[pos]] != 0) << (pos & 31); }
        V[w * Cs + lc] = word;
      }
      ser_col_build_pre(V + lc, PRE + lc, Cs, W);
    }
    __syncthreads();
    cl_rebuild_hard(sm, N, Mc, Cs);
    __syncthreads();

    const double *tape = nullptr;
    long long tape_len = 0;
    if (p.mode == SER_MODE_REPLAY) {
      tape = p.tape + p.tape_off[chain];
      tape_len = (long long)(p.tape_off[chain + 1] - p.tape_off[chain]);
    }
    SerWeights wt;
    wt.eps = p.eps; wt.H = sm.H; wt.hmax = 0;
    set_weights(wt, sc.c, sc.cc, sc.d, sc.dd);
    SerHard hd;
    hd.hcol = V + Mc; hd.hpre = PRE + Mc; hd.hp = sm.hp; hd.C = Cs; hd.W = W; hd.N = N; hd.nh = p.nh;
    hd.rank_tab = sm.hrank; hd.nonhard_tab = sm.nhpos;
    PropState ps;
    ps.k = 0; ps.buf = 0;

    for (int call = 0; call < p.n_calls && !(sc.flags & 1); call++) {
      const bool sampling = call >= p.burn_calls;
      for (int s = 0; s < p.sweeps_per_call; s++) {
        /* ================= stage this sweep's draws (every CTA its own copy) ================= */
        __syncthreads();
        PHASE_T0();
        if (p.mode == SER_MODE_REPLAY) {
          const long long need = sc.cursor + 6 + 2 * (long long)M;
          if (need > tape_len) { sc.flags |= 1; break; } /* uniform over the cluster */
          if (tid < 6) sm.draws_cd[tid] = tape[sc.cursor + tid];
          for (int t = tid; t < SER_PI_DRAWS; t += C) {
            const long long idx = need + t;
            const double u = idx < tape_len ? tape[idx] : 0.5;
            sm.draws_pi[t] = u; sm.logdraw[t] = log(u);
          }
        } else {
          if (tid < 4) {
            const int cnt = tid == 0 ? sc.f1a : tid == 1 ? sc.t0a : tid == 2 ? sc.f0a : sc.t1a;
            const double g = ser_gamma_ge1(1.0 + (double)cnt, p.seed, gchain, sc.sweep, (uint32_t)tid);
            const double go = __shfl_xor_sync(0xfu, g, 1);
            if (tid == 0 || tid == 2) {
              const double y = ser_beta_from_gammas(g, go);
              double val = tid == 0 ? sc.c : sc.d, l1m = tid == 0 ? sc.cc : sc.dd;
              const double lo = tid == 0 ? SER_MINC : SER_MIND, hi = tid == 0 ? SER_MAXC : SER_MAXD;
              if (y > 0.0) {
                const double ly = ser_log(y);
                if (lo <= ly && ly <= hi) { val = ly; l1m = ser_log(SER_SUB(1.0, ser_exp(ly))); }
              }
              sm.draws_cd[tid] = val; sm.draws_cd[tid + 1] = l1m;
            }
          }
          for (int t = tid; t < SER_PI_DRAWS; t += C) {
            const double u = ser_stream_uniform(p.seed, gchain, sc.sweep, SER_BLK_PI, (uint32_t)t);
            sm.draws_pi[t] = u; sm.logdraw[t] = log(ser_pos(u));
          }
        }
        __syncthreads();
        if (p.mode == SER_MODE_REPLAY) {
          const double yc = sm.draws_cd[0], lyc = sm.draws_cd[1], l1c = sm.draws_cd[2];
          const double yd = sm.draws_cd[3], lyd = sm.draws_cd[4], l1d = sm.draws_cd[5];
          if (yc > 0.0 && SER_MINC <= lyc && lyc <= SER_MAXC) { sc.c = lyc; sc.cc = l1c; }
          if (yd > 0.0 && SER_MIND <= lyd && lyd <= SER_MAXD) { sc.d = lyd; sc.dd = l1d; }
        } else {
          sc.c = sm.draws_cd[0]; sc.cc = sm.draws_cd[1]; sc.d = sm.draws_cd[2]; sc.dd = sm.draws_cd[3];
        }
        set_weights(wt, sc.c, sc.cc, sc.d, sc.dd);
        sc.counters[0]++; sc.counters[1]++;
        wt.hmax = ser_hmax(wt.g, N);
        for (int m = tid; m <= wt.hmax; m += C) sm.H[m] = ser_h_entry(wt.g, m);

        /* ================= a/b Gibbs of the local columns, one column group at a time (CTA-local: no cluster barrier) ======= */
        int changed = 0;
#pragma unroll 1
        for (int g = 0; g < ng; g++) {
          const int c0 = grp[2 * g], e0 = grp[2 * g + 1], c1 = grp[2 * g + 2], e1 = grp[2 * g + 3], nc = c1 - c0;
          int lpc = 1, lsh = 0;
          while (lpc < 8 && nc * lpc * 2 <= C) { lpc <<= 1; lsh++; }
          const int units = nc << lsh, sub = tid & (lpc - 1);
          __syncthreads(); /* previous group is done with pos / val; first group: publishes H */
          PHASE_MARK(0);
          { /* postings: a unit = (run of wq words, column) */
            const int wq = (W + lpc - 1) >> lsh;
            for (int u = tid; u < units; u += C) {
              const int cl = u >> lsh, qq = u & (lpc - 1), c = c0 + cl, w0 = qq * wq, w1 = min(W, w0 + wq);
              const int off_c = p.cl_off[c * R + rank] - e0;
              if (qq == 0) { sm.goff[cl] = off_c; sm.gones[cl] = (uint16_t)p.ones[c * R + rank]; }
              if (w0 < w1) {
                uint16_t *out = sm.pos + off_c + (int)PRE[w0 * Cs + c];
                for (int w = w0; w < w1; w++) {
                  uint32_t v = V[w * Cs + c];
                  while (v) { *out++ = (uint16_t)(32 * w + SER_FFS(v) - 1); v &= v - 1u; }
                }
              }
            }
          }
          __syncthreads();
          PHASE_MARK(1);
#pragma unroll 1
          for (int step = 0; step < 2; step++) {
            for (int ub = 0; ub < units; ub += C) { /* geometry + maximum; every item's log-weight stays in val */
              const int u = ub + tid;
              const bool live = u < units;
              const int cl = live ? (u >> lsh) : 0, c = c0 + cl;
              const SerStep st = step == 0 ? ser_step_a(V + c, PRE + c, Cs, W, N, sm.a16[c], sm.b16[c])
                                           : ser_step_b(V + c, PRE + c, Cs, W, N, sm.a16[c], sm.b16[c]);
              const uint16_t *pos = sm.pos + sm.goff[cl];
              double lm = -1.0e300;
              if (live) {
                double *Lc = sm.val + sm.goff[cl];
                for (int kk = sub; kk <= st.kb; kk += lpc) {
                  int q, n;
                  const double L = ser_item_eval(wt, st, pos, kk, &q, &n);
                  Lc[kk] = L;
                  lm = ser_fmax(lm, L);
                }
              }
              for (int o = lpc >> 1; o > 0; o >>= 1) lm = ser_fmax(lm, __shfl_xor_sync(0xffffffffu, lm, o));
              if (live && sub == 0) {
                sm.lmax[cl] = lm;
                *reinterpret_cast<uint2 *>(sm.st4 + 4 * cl) =
                    make_uint2((uint32_t)st.cur | ((uint32_t)st.bound << 16), (uint32_t)st.ocur | ((uint32_t)st.kb << 16));
              }
            }
            __syncthreads();
            PHASE_MARK(2);
            uint32_t ck_next = e0 + tid < e1 ? items[e0 + tid] : 0u;
            for (int e = e0 + tid; e < e1; e += C) { /* log-weight -> run weight, in place */
              const uint32_t ck = ck_next;
              if (e + C < e1) ck_next = items[e + C];
              const int cl = (int)(ck >> 16) - c0, kk = (int)(ck & 0xffffu);
              const int kb = (int)sm.st4[4 * cl + 3];
              if (kk <= kb) {
                const uint16_t *pos = sm.pos + (e - kk - e0);
                const int nones = (int)sm.gones[cl], bound = (int)sm.st4[4 * cl + 1];
                int q, qprev;
                if (step) { q = kk < kb ? N - 1 - (int)pos[nones - 1 - kk] : bound; qprev = kk > 0 ? N - 1 - (int)pos[nones - kk] : -1; }
                else { q = kk < kb ? (int)pos[kk] : bound; qprev = kk > 0 ? (int)pos[kk - 1] : -1; }
                sm.val[e - e0] = ser_item_weight_cached<1>(wt, sm.val[e - e0], q - qprev, sm.lmax[cl]);
              }
            }
            __syncthreads();
            PHASE_MARK(3);
            for (int ub = 0; ub < units; ub += C) { /* chunk sums, scan over the column's lanes, the item the uniform falls into */
              const int u = ub + tid;
              const bool live = u < units;
              const int cl = live ? (u >> lsh) : 0, c = c0 + cl;
              const int kb = (int)sm.st4[4 * cl + 3];
              double *val = sm.val + sm.goff[cl];
              const int chunk = (kb + lpc) >> lsh, k0 = min(kb + 1, sub * chunk), k1 = min(kb + 1, k0 + chunk);
              double tot = 0.0;
              if (live) for (int kk = k0; kk < k1; kk++) { tot = SER_ADD(tot, val[kk]); val[kk] = tot; }
              double incl = tot;
              for (int o = 1; o < lpc; o <<= 1) {
                const double t = __shfl_up_sync(0xffffffffu, incl, o);
                if (sub >= o) incl = SER_ADD(incl, t);
              }
              const int lane = tid & 31;
              const double total = __shfl_sync(0xffffffffu, incl, lane | (lpc - 1));
              const double before = __shfl_up_sync(0xffffffffu, incl, 1);
              double u01 = 0.0;
              if (live && sub == 0) { /* the column's uniform for this step */
                const int taxon = p.order[c * R + rank];
                if (p.mode == SER_MODE_REPLAY) u01 = tape[sc.cursor + 6 + 2 * taxon + step];
                else {
                  uint32_t o[4];
                  ser_philox4x32_10((uint32_t)taxon, SER_BLK_AB, sc.sweep, 0u, p.seed, gchain, o);
                  u01 = step == 0 ? ser_u53(o[0], o[1]) : ser_u53(o[2], o[3]);
                }
              }
              u01 = __shfl_sync(0xffffffffu, u01, lane & ~(lpc - 1));
              const double base = sub ? before : 0.0, target = SER_MUL(u01, total);
              if (live && k0 < k1 && incl >= target && (sub == 0 || base < target)) {
                int lo = k0, hi = k1 - 1;
                while (lo < hi) {
                  const int mid = (lo + hi) >> 1;
                  if (SER_ADD(base, val[mid]) >= target) hi = mid; else lo = mid + 1;
                }
                sm.pick16[cl] = (uint16_t)lo;
                sm.dsl[cl] = SER_SUB(target, lo > k0 ? SER_ADD(base, val[lo - 1]) : base);
              }
            }
            __syncthreads();
            PHASE_MARK(7);
            for (int cl = tid; cl < nc; cl += C) { /* closed-form pick inside the item's run */
              const int c = c0 + cl;
              const uint2 g4 = *reinterpret_cast<const uint2 *>(sm.st4 + 4 * cl);
              SerStep st;
              st.cur = (int)(g4.x & 0xffffu); st.bound = (int)(g4.x >> 16); st.ocur = (int)(g4.y & 0xffffu); st.kb = (int)(g4.y >> 16);
              st.nones = sm.gones[cl]; st.N = N; st.rev = step;
              int q, n;
              const double le = SER_SUB(ser_item_eval(wt, st, sm.pos + sm.goff[cl], (int)sm.pick16[cl], &q, &n), sm.lmax[cl]);
              const int pick = q - n + 1 + ser_run_pick<1>(wt, n, le, 0.0, sm.dsl[cl]);
              if (step == 0) { changed += pick != sm.a16[c]; sm.a16[c] = (uint16_t)pick; }
              else { changed += (N - pick) != sm.b16[c]; sm.b16[c] = (uint16_t)(N - pick); }
            }
            __syncthreads(); /* the b-step's geometry is computed under a different column -> thread map */
            PHASE_MARK(4);
          }
        }
        __syncthreads();
        const bool exact = sampling && s == p.sweeps_per_call - 1;
        if (exact) cluster.sync(); /* rank 0 is done with its item buffer before anybody stores terms into it */
        {
          int t1 = 0, len = 0, T1, LEN, CH;
          for (int lc = tid; lc < nloc; lc += C) {
            const int t1c = ser_col_popc(V + lc, PRE + lc, Cs, sm.a16[lc], sm.b16[lc]), lenc = sm.b16[lc] - sm.a16[lc];
            t1 += t1c; len += lenc;
            if (exact) { /* mcmc_logl's per-taxon term, mcmc.c:643-644, gathered in rank 0 */
              const int gc = lc * R + rank, f1 = p.ones[gc] - t1c, f0 = lenc - t1c, t0 = N - lenc - f1;
              TERMS0[p.order[gc]] = SER_ADD(SER_ADD(SER_ADD(SER_MUL((double)t0, wt.cc), SER_MUL((double)f0, wt.d)), SER_MUL((double)t1c, wt.dd)),
                                            SER_MUL((double)f1, wt.c));
            }
          }
          cluster_sum3(cluster, sm, R, rank, t1, len, changed, ps.buf, &T1, &LEN, &CH);
          totals_from(p, wt, T1, LEN, &sc.t0a, &sc.f0a, &sc.t1a, &sc.f1a, &sc.loglik);
          sc.counters[2] += CH;
          if (exact) sc.loglik = cluster_sequential_sum(cluster, sm, R, rank, M);
        }

        PHASE_MARK(5);
        /* ================= 16 proposals for pi: decoded by every CTA, deltas of the local columns, one exchange each ======= */
        ps.k = 0;
        for (int prop = 0; prop < 16; prop++) {
          const int kind = prop == 0 ? 3 : ((prop - 1) % 3);
          int dt0 = 0, dt1 = 0, nz = 0, D0, D1;
          double delta;
          if (kind == 0) { /* pi1 */
            const int i = ser_draw_int(sm.draws_pi[ps.k], N);
            int j = ser_draw_int(sm.draws_pi[ps.k + 1], N - 1);
            ps.k += 2;
            if (j >= i) j++;
            const int lo = min(i, j), hi = max(i, j);
            if (ser_is_hard(hd, i) && ser_hard_count(hd, lo, hi) > 1) continue;
            auto redo = [&](int lc, int *x0, int *x1) { ser_pi1_delta(V + lc, Cs, sm.a16[lc], sm.b16[lc], i, j, x0, x1); };
            for (int lc = tid; lc < nloc; lc += C) { int x0, x1; redo(lc, &x0, &x1); dt0 += x0; dt1 += x1; nz |= (x0 | x1) != 0; }
            if (!mh_decide_cl(cluster, p, sm, wt, ps, R, rank, nloc, dt0, dt1, nz, exact, &D0, &D1, &delta, redo)) continue;
            for (int lc = tid; lc <= Mc; lc += C) {
              if (lc < nloc) { int a = sm.a16[lc], b = sm.b16[lc]; ser_pi1_apply_ab(&a, &b, i, j); sm.a16[lc] = (uint16_t)a; sm.b16[lc] = (uint16_t)b; }
              if (lc < nloc || lc == Mc) ser_col_rotate(V + lc, Cs, W, i, j, PRE + lc);
            }
            for (int n = lo + tid; n <= hi; n += C) sm.tmp16[n] = sm.rpi[i < j ? (n < j ? n + 1 : i) : (n > j ? n - 1 : i)];
            __syncthreads();
            for (int n = lo + tid; n <= hi; n += C) sm.rpi[n] = sm.tmp16[n];
            cl_rebuild_hard(sm, N, Mc, Cs);
            sc.counters[3]++;
          } else if (kind == 1 || kind == 3) { /* pi2 */
            int i, j;
            if (kind == 1) {
              i = ser_draw_int(sm.draws_pi[ps.k], N);
              j = ser_draw_int(sm.draws_pi[ps.k + 1], N - 1);
              ps.k += 2;
              if (j >= i) j++;
              else { const int t = i; i = j; j = t; }
            } else {
              i = ser_draw_int(sm.draws_pi[ps.k], N - 1);
              ps.k += 1;
              j = i + 1;
            }
            if (ser_hard_count(hd, i, j) > 1) continue;
            const int inc1 = ser_draw_int(sm.draws_pi[ps.k], 2), inc2 = ser_draw_int(sm.draws_pi[ps.k + 1], 2);
            ps.k += 2;
            auto redo = [&](int lc, int *x0, int *x1) { ser_pi2_delta(V + lc, PRE + lc, Cs, sm.a16[lc], sm.b16[lc], i, j, inc1, inc2, x0, x1); };
            for (int lc = tid; lc < nloc; lc += C) { int x0, x1; redo(lc, &x0, &x1); dt0 += x0; dt1 += x1; nz |= (x0 | x1) != 0; }
            if (!mh_decide_cl(cluster, p, sm, wt, ps, R, rank, nloc, dt0, dt1, nz, exact, &D0, &D1, &delta, redo)) continue;
            for (int lc = tid; lc <= Mc; lc += C) {
              if (lc < nloc) {
                int a = sm.a16[lc], b = sm.b16[lc];
                const int ain = ser_in_window(a, i, j + 1, inc1, inc2), bin = ser_in_window(b, i, j + 1, inc1, inc2);
                ser_mirror_ab(a, b, ain, bin, i + j + 1, &a, &b);
                sm.a16[lc] = (uint16_t)a; sm.b16[lc] = (uint16_t)b;
              }
              if (lc < nloc || lc == Mc) ser_col_reverse(V + lc, Cs, W, i, j, PRE + lc);
            }
            for (int n = i + tid; n <= j; n += C) sm.tmp16[n] = sm.rpi[i + j - n];
            __syncthreads();
            for (int n = i + tid; n <= j; n += C) sm.rpi[n] = sm.tmp16[n];
            cl_rebuild_hard(sm, N, Mc, Cs);
            sc.counters[kind == 1 ? 4 : 5]++;
          } else { /* pi3 */
            const int nfree = N - p.nh;
            if (nfree < 2) continue;
            const int r1 = ser_draw_int(sm.draws_pi[ps.k], nfree), r2 = ser_draw_int(sm.draws_pi[ps.k + 1], nfree - 1);
            ps.k += 2;
            int ir, jr;
            if (r1 <= r2) { ir = r1; jr = r2 + 1; } else { ir = r2; jr = r1; }
            const SerPi3 g = ser_pi3_window(hd, ir, jr);
            const int inc1 = ser_draw_int(sm.draws_pi[ps.k], 2), inc2 = ser_draw_int(sm.draws_pi[ps.k + 1], 2);
            ps.k += 2;
            const bool hb = p.nh <= 32;
            auto redo = [&](int lc, int *x0, int *x1) {
              if (hb) ser_pi3_delta<true>(V + lc, PRE + lc, Cs, hd, g, sm.a16[lc], sm.b16[lc], inc1, inc2, x0, x1, sm.hb32[lc]);
              else ser_pi3_delta<false>(V + lc, PRE + lc, Cs, hd, g, sm.a16[lc], sm.b16[lc], inc1, inc2, x0, x1);
            };
            for (int lc = tid; lc < nloc; lc += C) { int x0, x1; redo(lc, &x0, &x1); dt0 += x0; dt1 += x1; nz |= (x0 | x1) != 0; }
            if (!mh_decide_cl(cluster, p, sm, wt, ps, R, rank, nloc, dt0, dt1, nz, exact, &D0, &D1, &delta, redo)) continue;
            for (int n = g.i + tid; n <= g.j; n += C) sm.perm16[n] = (uint16_t)ser_pi3_perm(hd, g, n);
            __syncthreads();
            for (int lc = tid; lc < nloc; lc += C) {
              int a = sm.a16[lc], b = sm.b16[lc];
              const int ain = ser_in_window(a, g.i, g.j + 1, inc1, inc2), bin = ser_in_window(b, g.i, g.j + 1, inc1, inc2);
              ser_mirror_ab(a, b, ain, bin, g.i + g.j + 1, &a, &b);
              sm.a16[lc] = (uint16_t)a; sm.b16[lc] = (uint16_t)b;
              ser_col_permute(V + lc, Cs, W, g.i, g.j, sm.perm16, PRE + lc);
            }
            for (int n = g.i + tid; n <= g.j; n += C) sm.tmp16[n] = sm.rpi[sm.perm16[n]];
            __syncthreads();
            for (int n = g.i + tid; n <= g.j; n += C) sm.rpi[n] = sm.tmp16[n];
            sc.counters[6]++;
          }
          sc.t0a += D0; sc.f0a -= D0; sc.t1a += D1; sc.f1a -= D1;
          sc.loglik = SER_ADD(sc.loglik, delta);
          __syncthreads();
        }

        if (p.mode == SER_MODE_REPLAY) sc.cursor += 6 + 2 * (long long)M + ps.k;
        else sc.sweep++;
        sc.counters[7]++;
        PHASE_MARK(6);
      }
      if (sc.flags & 1) break;

      if (sampling) { /* thinned sample: the site order by rank 0, a / b by the columns' owners */
        const int sidx = sc.n_samples - p.sample_base;
        if (sidx < p.max_samples) {
          const size_t row = (size_t)chain * p.max_samples + sidx;
          if (p.store >= SER_STORE_PI && rank == 0)
            for (int pos = tid; pos < N; pos += C) p.samp_pi[row * N + sm.rpi[pos]] = (uint16_t)pos;
          if (p.store >= SER_STORE_FULL) {
            for (int lc = tid; lc < nloc; lc += C) {
              const int taxon = p.order[lc * R + rank];
              p.samp_a[row * M + taxon] = sm.a16[lc]; p.samp_b[row * M + taxon] = sm.b16[lc];
            }
            if (tid == 0 && rank == 0) { p.samp_cdl[row * 3 + 0] = sc.c; p.samp_cdl[row * 3 + 1] = sc.d; p.samp_cdl[row * 3 + 2] = sc.loglik; }
          }
        }
        sc.sum_negll = SER_ADD(sc.sum_negll, -sc.loglik);
        sc.sum_ec = SER_ADD(sc.sum_ec, exp(sc.c));
        sc.sum_ed = SER_ADD(sc.sum_ed, exp(sc.d));
        sc.n_samples++;
      }
    }

    __syncthreads();
    for (int lc = tid; lc < nloc; lc += C) {
      p.ab[(size_t)chain * 2 * p.Mpad + lc * R + rank] = sm.a16[lc];
      p.ab[(size_t)chain * 2 * p.Mpad + p.Mpad + lc * R + rank] = sm.b16[lc];
    }
    if (rank == 0) {
      for (int n = tid; n < N; n += C) p.rpi[(size_t)chain * p.Npad + n] = sm.rpi[n];
      if (tid == 0) p.scal[chain] = sc;
    }
  }
  cluster.sync(); /* nobody leaves while its shared memory may still be written */
}
