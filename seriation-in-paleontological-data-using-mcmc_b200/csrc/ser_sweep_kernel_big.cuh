/* ser_sweep_kernel_big.cuh -- the large-shape sweep kernel: persistent CTAs, columns in a global scratch slot, Gibbs phase staged through shared memory
 * (warp batches: one warp serves a few columns on its own; or CTA-wide column groups).
 * Part of the single translation unit ser_kernels.cu (included there, in this order). */

/* ------------------------------------------------------------------ the sweep kernel, large shapes
 * Same algorithm and building blocks as ser_sweep_kernel, for matrices whose bit columns, prefix
 * tables and item buffers exceed shared memory (e.g. 1024 sites x 4096 taxa: 0.7 MB + 0.3 MB +
 * 3.2 MB per chain).  A CTA owns a slot of L2-resident global scratch and walks over chains
 * (persistent grid); every thread owns the columns tid, tid+C, ...; a/b live in shared memory. */
struct BigSmem {
  double *draws_pi, *logdraw, *draws_cd, *H;
  double *lmax; /* gcap: per column of the running group */
  double *val;  /* icap: item weights / cumulative weights of the running group */
  int *red;
  uint16_t *a16, *b16, *hp, *rpi, *tmp16, *perm16;
  uint16_t *st4; /* 4 * gcap */
  uint16_t *gones; /* gcap: ones of the running group's columns */
  int *goff;       /* gcap: first item of each column relative to the group's first item */
  uint16_t *pos; /* icap: postings of the running group's columns */
  double *uab;              /* 2 gcap: the two uniforms (a-step, b-step) of every column of the running group */
  double *wcol;             /* manycd: 4 gcap per-column weights A, g, 1/g, 1/(1-e^-g) of the running group */
  double *redd;             /* manycd: 2 x 32 doubles of reduction scratch */
  uint32_t *hcol;           /* W: the hard-site mask in position order (stride 1; never leaves shared memory) */
  uint16_t *hpre;           /* W+1: its prefix table */
  uint16_t *hrank, *nhpos;  /* N+2 each: SerHard's tables */
  int *bctr;                /* next column batch of the running sweep (warp-batch Gibbs phase) */
};
/* what one team of the Gibbs phase works in: the whole group-local arrays (team = CTA) or a warp's slices of them */
struct BigTeam {
  uint16_t *pos; double *val; int cap;
  int *goff; uint16_t *gones; double *lmax; uint16_t *st4; double *uab; double *wcol;
};
/* gcap = columns of the widest CTA-wide group (0 with warp batches, which keep the per-column values in registers);
 * wcols = columns the per-taxon weights are staged for (manycd: gcap, or 32 per warp with warp batches) */
__host__ __device__ inline size_t big_layout(BigSmem *s, unsigned char *base, int N, int M, int icap, int gcap, int manycd, int wcols)
{
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 15) & ~(size_t)15; return o; };
  size_t o_dp = take(8 * SER_PI_DRAWS), o_ld = take(8 * SER_PI_DRAWS), o_dc = take(8 * 8), o_H = take(8 * (size_t)(N + 2 < SER_HCAP ? N + 2 : SER_HCAP));
  size_t o_go = take(4 * (size_t)gcap), o_gn = take(2 * (size_t)gcap), o_lm = take(8 * (size_t)gcap), o_val = take(8 * (size_t)icap), o_r = take(sizeof(int) * 2 * SER_MAX_WARPS * 4);
  size_t o_a = take(2 * (size_t)M), o_b = take(2 * (size_t)M), o_st = take(2 * 4 * (size_t)gcap), o_hp = take(2 * (size_t)(N + 1));
  size_t o_p = take(2 * (size_t)N), o_q = take(2 * (size_t)N), o_m = take(2 * (size_t)N), o_pos = take(2 * (size_t)icap);
  size_t o_hc = take(4 * (size_t)(N / 32 + 1)), o_hq = take(2 * (size_t)(N / 32 + 2)), o_ua = take(16 * (size_t)gcap);
  size_t o_wc = take(manycd ? 32 * (size_t)wcols : 0), o_rd = take(manycd ? 8 * 2 * SER_MAX_WARPS : 0);
  size_t o_hr = take(2 * (size_t)(N + 2)), o_nh = take(2 * (size_t)(N + 2)), o_bc = take(16);
  if (s) {
    s->bctr = (int *)(base + o_bc);
    s->uab = (double *)(base + o_ua); s->wcol = (double *)(base + o_wc); s->redd = (double *)(base + o_rd);
    s->hcol = (uint32_t *)(base + o_hc); s->hpre = (uint16_t *)(base + o_hq);
    s->hrank = (uint16_t *)(base + o_hr); s->nhpos = (uint16_t *)(base + o_nh);
    s->val = (double *)(base + o_val); s->pos = (uint16_t *)(base + o_pos);
    s->goff = (int *)(base + o_go); s->gones = (uint16_t *)(base + o_gn);
    s->draws_pi = (double *)(base + o_dp); s->logdraw = (double *)(base + o_ld); s->draws_cd = (double *)(base + o_dc);
    s->H = (double *)(base + o_H); s->lmax = (double *)(base + o_lm); s->red = (int *)(base + o_r);
    s->a16 = (uint16_t *)(base + o_a); s->b16 = (uint16_t *)(base + o_b); s->st4 = (uint16_t *)(base + o_st);
    s->hp = (uint16_t *)(base + o_hp); s->rpi = (uint16_t *)(base + o_p); s->tmp16 = (uint16_t *)(base + o_q);
    s->perm16 = (uint16_t *)(base + o_m);
  }
  return off;
}

/* per-column weights (manycd): c, log(1-e^c), d, log(1-e^d) of sorted column col from the chain's cd4 rows */
__device__ __forceinline__ void big_col_weights(const double *cd4, int Mpad, int col, SerWeights *w)
{
  w->c = cd4[col]; w->cc = cd4[Mpad + col]; w->d = cd4[2 * Mpad + col]; w->dd = cd4[3 * Mpad + col];
}

/* MH tail for the large-shape kernel: the thread's deltas are already summed over its columns (`tsum` = its float
 * terms, per-taxon c, d only); the degenerate / exact cases re-evaluate the per-taxon deltas through `redo` (a lambda)
 * and add the terms in taxon order (see mh_decide) */
template <bool MANY, typename Redo>
__device__ __forceinline__ bool mh_decide_big(const KParams &p, const BigSmem &sm, const SerWeights &wt, const double *cd4, PropState &ps,
                                              double *terms, int dt0, int dt1, int nz, double tsum, bool exact, int *D0, int *D1,
                                              double *delta_out, Redo redo)
{
  int NZ;
  double delta = 0.0;
  if constexpr (MANY) block_sum3d(dt0, dt1, nz, tsum, sm.red, sm.redd, ps.buf, D0, D1, &NZ, &delta);
  else block_sum3(dt0, dt1, nz, sm.red, ps.buf, D0, D1, &NZ);
  auto reference_sum = [&]() {
    double acc = 0.0;
    __syncthreads();
    for (int c = threadIdx.x; c < p.M; c += blockDim.x) {
      int x0, x1;
      redo(c, &x0, &x1);
      if constexpr (MANY) { SerWeights w; big_col_weights(cd4, p.Mpad, c, &w); terms[p.order[c]] = ser_term(w, x0, x1); }
      else terms[p.order[c]] = ser_term(wt, x0, x1);
    }
    __syncthreads();
    if (threadIdx.x < 32) { /* one warp walks the dependent chain, the others wait (see sequential_term_sum) */
      for (int m = 0; m < p.M; m++) acc = SER_ADD(acc, terms[m]);
      if (threadIdx.x == 0) sm.draws_cd[7] = acc;
    }
    __syncthreads();
    return sm.draws_cd[7];
  };
  bool seq = false;
  if constexpr (MANY) {
    if (!NZ) delta = 0.0;
    else if (fabs(delta) < 1e-7) { delta = reference_sum(); seq = true; }
  } else {
    if (*D0 == 0 && *D1 == 0) {
      delta = 0.0;
      if (NZ) { delta = reference_sum(); seq = true; }
    } else {
      delta = ser_term(wt, *D0, *D1);
    }
  }
  bool accept = delta >= 0.0;
  if (!accept) accept = delta > sm.logdraw[ps.k++];
  if (accept && exact && !seq && NZ) delta = reference_sum();
  *delta_out = delta;
  return accept;
}

/* the hard-site tables from the shared-memory copy of the hard mask (as rebuild_hard) */
__device__ __forceinline__ void big_rebuild_hard(const BigSmem &sm, int N)
{
  for (int q = threadIdx.x; q <= N; q += blockDim.x) {
    const int r = ser_rank1(sm.hcol, sm.hpre, 1, q);
    sm.hrank[q] = (uint16_t)r;
    if (q < N) {
      if ((sm.hcol[q >> 5] >> (q & 31)) & 1u) sm.hp[r] = (uint16_t)q;
      else sm.nhpos[q - r] = (uint16_t)q;
    }
  }
}

/* MANY = per-taxon c, d (manycd = 1, mcmc.c:777-785, :807-815): the chain's cd4 rows in HBM hold every column's c, log(1-e^c),
 * d, log(1-e^d); the weights of a group's columns are staged in shared memory, geometric run sums are evaluated on the fly,
 * delta / loglik are float sums over taxa (mh_decide_big). */
template <bool MANY, bool WB>
__global__ void __launch_bounds__(1024, 1) ser_sweep_kernel_big(KParams p)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  BigSmem sm;
  __shared__ unsigned int s_gchain;
  big_layout(&sm, smem_raw, p.N, p.M, p.big_icap, p.big_gcap, MANY ? 1 : 0, WB ? (int)blockDim.x : p.big_gcap);
  const int tid = threadIdx.x, N = p.N, M = p.M, C = blockDim.x, W = p.W, Cs = p.Cs;
  constexpr int BG = SER_BIG_G;
  uint32_t *V = p.gV + (size_t)blockIdx.x * W * Cs;
  uint16_t *PRE = p.gpre + (size_t)blockIdx.x * ((W >> BG) + 1) * Cs; /* one prefix count per 2^BG words (ser_pre_at) */
  double *TERMS = sm.val; /* per-taxon terms of the exact sums: the item-weight buffer is idle outside the Gibbs phase (icap >= M) */
  if (WB && tid == 0) *sm.bctr = 0;

  for (int chain = blockIdx.x; chain < p.n_chains; chain += gridDim.x) {
    const unsigned int &gchain = s_gchain; /* in shared memory, like ser_sweep_kernel's */
    double *cd4 = MANY ? p.cd4 + (size_t)chain * 4 * p.Mpad : nullptr;
    __syncthreads(); /* previous chain's state fully saved before the scratch is reused */
    if (threadIdx.x == 0) s_gchain = global_chain(p, chain); /* visible after the next barrier */
    ChainScalars sc = p.scal[chain];
    for (int n = tid; n < N; n += C) sm.rpi[n] = p.rpi[(size_t)chain * p.Npad + n];
    for (int c = tid; c < M; c += C) {
      sm.a16[c] = p.ab[(size_t)chain * 2 * p.Mpad + c];
      sm.b16[c] = p.ab[(size_t)chain * 2 * p.Mpad + p.Mpad + c];
    }
    __syncthreads();
    /* position-ordered columns + prefix tables of the owned columns */
    for (int c = tid; c <= M; c += C) {
      for (int w = 0; w < W; w++) {
        uint32_t word = 0;
        const int pend = min(32 * w + 32, N);
        if (c < M) { for (int pos = 32 * w; pos < pend; pos++) word |= (uint32_t)cell(p, sm.rpi, pos, c) << (pos & 31); V[w * Cs + c] = word; }
        else { for (int pos = 32 * w; pos < pend; pos++) word |= (uint32_t)(p.hard[sm.rpi[pos]] != 0) << (pos & 31); sm.hcol[w] = word; }
      }
      if (c < M) ser_col_build_pre<BG>(V + c, PRE + c, Cs, W);
      else ser_col_build_pre(sm.hcol, sm.hpre, 1, W);
    }
    __syncthreads();
    big_rebuild_hard(sm, N);
    __syncthreads();

    const double *tape = nullptr;
    long long tape_len = 0;
    if (p.mode == SER_MODE_REPLAY) {
      tape = p.tape + p.tape_off[chain];
      tape_len = (long long)(p.tape_off[chain + 1] - p.tape_off[chain]);
    }
    SerWeights wt;
    wt.eps = p.eps; wt.H = sm.H; wt.hmax = MANY ? N + 1 : 0; /* MANY: geometric sums on the fly, no table bound */
    set_weights(wt, sc.c, sc.cc, sc.d, sc.dd);
    SerHard hd;
    hd.hcol = sm.hcol; hd.hpre = sm.hpre; hd.hp = sm.hp; hd.C = 1; hd.W = W; hd.N = N; hd.nh = p.nh; hd.rank_tab = sm.hrank; hd.nonhard_tab = sm.nhpos;
    PropState ps;
    ps.k = 0; ps.buf = 0;

    for (int call = 0; call < p.n_calls && !(sc.flags & 1); call++) {
      const bool sampling = call >= p.burn_calls; /* burn-in calls first, then sampling calls */
      for (int s = 0; s < p.sweeps_per_call; s++) {
        /* ================= stage this sweep's draws ================= */
        __syncthreads();
        PHASE_T0();
        if constexpr (MANY) {
          /* M Betas for c, M for d (mcmc.c:777-785, :807-815), the pi draws; the a/b uniforms are staged per column group */
          if (p.mode == SER_MODE_REPLAY) {
            const long long need = sc.cursor + 8 * (long long)M;
            if (need > tape_len) { sc.flags |= 1; break; }
            for (int t = tid; t < SER_PI_DRAWS; t += C) {
              const long long idx = need + t;
              const double u = idx < tape_len ? tape[idx] : 0.5;
              sm.draws_pi[t] = u; sm.logdraw[t] = log(u);
            }
          } else {
            for (int t = tid; t < SER_PI_DRAWS; t += C) {
              const double u = ser_stream_uniform(p.seed, gchain, sc.sweep, SER_BLK_PI, (uint32_t)t);
              sm.draws_pi[t] = u; sm.logdraw[t] = log(ser_pos(u));
            }
          }
          for (int c = tid; c < M; c += C) { /* Beta(1+f1_m, 1+t0_m) and Beta(1+f0_m, 1+t1_m) from the taxon's own counts */
            const int taxon = p.order[c];
            double yc = 0.0, lyc = 0.0, l1c = 0.0, yd = 0.0, lyd = 0.0, l1d = 0.0;
            if (p.mode == SER_MODE_REPLAY) {
              const double *tc = tape + sc.cursor + 3 * taxon, *td = tape + sc.cursor + 3 * (long long)M + 3 * taxon;
              yc = tc[0]; lyc = tc[1]; l1c = tc[2];
              yd = td[0]; lyd = td[1]; l1d = td[2];
            } else {
              const int t1 = ser_col_popc<BG>(V + c, PRE + c, Cs, sm.a16[c], sm.b16[c]), len = sm.b16[c] - sm.a16[c];
              const int f1 = p.ones[c] - t1, f0 = len - t1, t0 = N - len - f1;
              const uint32_t blk = SER_BLK_MANYCD + 4u * (uint32_t)taxon;
              yc = ser_beta_from_gammas(ser_gamma_ge1(1.0 + (double)f1, p.seed, gchain, sc.sweep, blk),
                                        ser_gamma_ge1(1.0 + (double)t0, p.seed, gchain, sc.sweep, blk + 1u));
              yd = ser_beta_from_gammas(ser_gamma_ge1(1.0 + (double)f0, p.seed, gchain, sc.sweep, blk + 2u),
                                        ser_gamma_ge1(1.0 + (double)t1, p.seed, gchain, sc.sweep, blk + 3u));
              if (yc > 0.0) { lyc = ser_log(yc); l1c = ser_log(SER_SUB(1.0, ser_exp(lyc))); }
              if (yd > 0.0) { lyd = ser_log(yd); l1d = ser_log(SER_SUB(1.0, ser_exp(lyd))); }
            }
            if (yc > 0.0 && SER_MINC <= lyc && lyc <= SER_MAXC) { cd4[c] = lyc; cd4[p.Mpad + c] = l1c; }
            if (yd > 0.0 && SER_MIND <= lyd && lyd <= SER_MAXD) { cd4[2 * p.Mpad + c] = lyd; cd4[3 * p.Mpad + c] = l1d; }
            if (taxon == 0) { sm.draws_cd[0] = cd4[c]; sm.draws_cd[1] = cd4[2 * p.Mpad + c]; }
          }
          sc.counters[0] += M; sc.counters[1] += M;
        } else {
          if (p.mode == SER_MODE_REPLAY) {
            const long long need = sc.cursor + 6 + 2 * (long long)M;
            if (need > tape_len) { sc.flags |= 1; break; }
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
          wt.hmax = min(ser_hmax(wt.g, N), SER_HCAP - 1);
          for (int m = tid; m <= wt.hmax; m += C) sm.H[m] = ser_h_entry(wt.g, m);

        }

        /* ================= a/b Gibbs, item formulation =================
         * Two forms (DESIGN.md 3.3): warp batches (WB, gibbs_warp below) and CTA-wide column groups (gibbs_team).
         *
         * CTA-wide groups, one column group at a time: the group's postings and item weights live in shared memory (icap
         * items), so the per-column loops run at shared-memory latency.  A column is served by `lpc` adjacent lanes (1..8, as
         * many as the block can spare for the group), which split its loops: the maximum is a lane-strided partial maximum +
         * shuffle, the cumulative weights are a per-lane serial sum over a contiguous chunk + a shuffle scan of the lane
         * totals.  Per group: postings; then for the a-step and the b-step: geometry + maximum, run weights (dense over the
         * group's items), scan + inverse CDF.  The body is written for a team of T threads with index t (T = the CTA here;
         * WARP = true, a team of one warp behind __syncwarp, was the first form of the warp batches). */
        int changed = 0;
        auto gibbs_team = [&](const BigTeam &TM, const int t, const int T, const int c0, const int e0, const int c1,
                              const int e1, const int lsh) {
          constexpr bool WARP = false;
          auto team_sync = [&]() { if constexpr (WARP) __syncwarp(); else __syncthreads(); };
          const int nc = c1 - c0, lpc = 1 << lsh;
          const int units = nc << lsh, sub = t & (lpc - 1);
          team_sync(); /* the team's previous columns are done with pos / val; first group: publishes H */
          PHASE_MARK(0);
          { /* postings: lane qq of a column's lpc lanes expands a run of wq words (a warp reads 32 / lpc consecutive
             * columns of lpc word rows: whole 32-byte sectors); the prefix table gives the lane's first slot.  Columns
             * map to lanes exactly as in the passes below, so what a column's lanes write here is read by the same warp. */
            const int wq = (W + lpc - 1) >> lsh;
            for (int u = t; u < units; u += T) {
              const int qq = u & (lpc - 1), cl = u >> lsh, c = c0 + cl, w0 = qq * wq, w1 = min(W, w0 + wq);
              /* every load of the unit is issued before the first one is needed */
              uint32_t vv[8];
#pragma unroll
              for (int k = 0; k < 8; k++) vv[k] = w0 + k < w1 ? V[(w0 + k) * Cs + c] : 0u;
              const int first = w0 < w1 ? ser_pre_at<BG>(V + c, PRE + c, Cs, w0) : 0, off_c = p.off[c] - e0;
              if (qq == 0) { TM.goff[cl] = off_c; TM.gones[cl] = (uint16_t)p.ones[c]; } /* the team's column table */
              uint16_t *out = TM.pos + off_c + first;
              for (int wb = w0; wb < w1; wb += 8) {
                if (wb > w0) {
#pragma unroll
                  for (int k = 0; k < 8; k++) vv[k] = wb + k < w1 ? V[(wb + k) * Cs + c] : 0u;
                }
#pragma unroll
                for (int k = 0; k < 8; k++) {
                  uint32_t v = vv[k];
                  while (v) { *out++ = (uint16_t)(32 * (wb + k) + SER_FFS(v) - 1); v &= v - 1u; }
                }
              }
            }
          }
          for (int cl = t; cl < nc; cl += T) { /* the two uniforms of every column of the team (mcmc.c:951, :963 -> :909) */
            const int taxon = p.order[c0 + cl];
            if (p.mode == SER_MODE_REPLAY) {
              const long long u0 = sc.cursor + (MANY ? 6 * (long long)M : 6) + 2 * taxon;
              TM.uab[2 * cl] = tape[u0]; TM.uab[2 * cl + 1] = tape[u0 + 1];
            }
            else {
              uint32_t o[4];
              ser_philox4x32_10((uint32_t)taxon, SER_BLK_AB, sc.sweep, 0u, p.seed, gchain, o);
              TM.uab[2 * cl] = ser_u53(o[0], o[1]); TM.uab[2 * cl + 1] = ser_u53(o[2], o[3]);
            }
            if constexpr (MANY) { /* the column's own weights for the passes of this group */
              SerWeights w;
              big_col_weights(cd4, p.Mpad, c0 + cl, &w);
              ser_set_weights_own(&w, w.c, w.cc, w.d, w.dd, N);
              TM.wcol[4 * cl + 0] = w.A; TM.wcol[4 * cl + 1] = w.g; TM.wcol[4 * cl + 2] = w.inv_g; TM.wcol[4 * cl + 3] = w.hs;
            }
          }
          if constexpr (MANY && !WARP) __syncthreads(); /* the columns' weights were staged by other threads */
          else __syncwarp();                            /* postings and column table: written and read by the same warp */
          PHASE_MARK(1);
#pragma unroll 1
          for (int step = 0; step < 2; step++) {
            for (int ub = 0; ub < units; ub += T) { /* warp-uniform trip count: the shuffles need every lane */
              const int u = ub + t;
              const bool live = u < units;
              const int cl = live ? (u >> lsh) : 0, c = c0 + cl;
              const SerStep st = step == 0 ? ser_step_a<BG>(V + c, PRE + c, Cs, W, N, sm.a16[c], sm.b16[c])
                                           : ser_step_b<BG>(V + c, PRE + c, Cs, W, N, sm.a16[c], sm.b16[c]);
              const uint16_t *pos = TM.pos + TM.goff[cl];
              double lm = -1.0e300;
              if (live) { /* every item's log-weight stays in val for the dense pass */
                double *Lc = TM.val + TM.goff[cl];
                SerWeights w = wt;
                if constexpr (MANY) { w.A = TM.wcol[4 * cl + 0]; w.g = TM.wcol[4 * cl + 1]; }
                for (int kk = sub; kk <= st.kb; kk += lpc) {
                  int q, n;
                  const double L = ser_item_eval(w, st, pos, kk, &q, &n);
                  Lc[kk] = L;
                  lm = ser_fmax(lm, L);
                }
              }
              for (int o = lpc >> 1; o > 0; o >>= 1) lm = ser_fmax(lm, __shfl_xor_sync(0xffffffffu, lm, o));
              if (live && sub == 0) {
                TM.lmax[cl] = lm;
                *reinterpret_cast<uint2 *>(TM.st4 + 4 * cl) =
                    make_uint2((uint32_t)st.cur | ((uint32_t)st.bound << 16), (uint32_t)st.ocur | ((uint32_t)st.kb << 16));
              }
            }
            team_sync();
            PHASE_MARK(2);
            uint32_t ck_next = e0 + t < e1 ? p.item_col[e0 + t] : 0u; /* fetched one iteration ahead */
            for (int e = e0 + t; e < e1; e += T) {
              const uint32_t ck = ck_next;
              if (e + T < e1) ck_next = p.item_col[e + T];
              const int cl = (int)(ck >> 16) - c0, kk = (int)(ck & 0xffffu);
              const int kb = (int)TM.st4[4 * cl + 3];
              if (kk <= kb) { /* log-weight -> run weight, in place; the run length from the postings */
                SER_CHECK(cl >= 0 && cl < nc && e - e0 < TM.cap && e - kk - e0 >= 0);
                const uint16_t *pos = TM.pos + (e - kk - e0);
                const int nones = (int)TM.gones[cl], bound = (int)TM.st4[4 * cl + 1];
                int q, qprev; /* ser_item_eval's q and qprev */
                if (step) { q = kk < kb ? N - 1 - (int)pos[nones - 1 - kk] : bound; qprev = kk > 0 ? N - 1 - (int)pos[nones - kk] : -1; }
                else { q = kk < kb ? (int)pos[kk] : bound; qprev = kk > 0 ? (int)pos[kk - 1] : -1; }
                if constexpr (MANY) {
                  SerWeights w = wt;
                  w.g = TM.wcol[4 * cl + 1]; w.inv_g = TM.wcol[4 * cl + 2]; w.hs = TM.wcol[4 * cl + 3];
                  TM.val[e - e0] = ser_item_weight_cached<0>(w, TM.val[e - e0], q - qprev, TM.lmax[cl]);
                } else {
                  TM.val[e - e0] = ser_item_weight_cached<1>(wt, TM.val[e - e0], q - qprev, TM.lmax[cl]);
                }
              }
            }
            team_sync();
            PHASE_MARK(3);
            for (int ub = 0; ub < units; ub += T) { /* chunk sums, scan over the column's lanes, the item the uniform falls into */
              const int u = ub + t;
              const bool live = u < units;
              const int cl = live ? (u >> lsh) : 0;
              const int kb = (int)TM.st4[4 * cl + 3];
              double *val = TM.val + TM.goff[cl];
              const int chunk = (kb + lpc) >> lsh, k0 = min(kb + 1, sub * chunk), k1 = min(kb + 1, k0 + chunk);
              double tot = 0.0;
              if (live) for (int kk = k0; kk < k1; kk++) { tot = SER_ADD(tot, val[kk]); val[kk] = tot; }
              double incl = tot; /* inclusive scan of the chunk totals over the column's lanes */
              for (int o = 1; o < lpc; o <<= 1) {
                const double tt = __shfl_up_sync(0xffffffffu, incl, o);
                if (sub >= o) incl = SER_ADD(incl, tt);
              }
              const int lane = t & 31;
              const double total = __shfl_sync(0xffffffffu, incl, lane | (lpc - 1));
              const double before = __shfl_up_sync(0xffffffffu, incl, 1);
              const double u01 = live ? TM.uab[2 * cl + step] : 0.0;
              const double base = sub ? before : 0.0, target = SER_MUL(u01, total);
              if (live && k0 < k1 && incl >= target && (sub == 0 || base < target)) { /* the first chunk that reaches the target */
                int lo = k0, hi = k1 - 1;
                while (lo < hi) {
                  const int mid = (lo + hi) >> 1;
                  if (SER_ADD(base, val[mid]) >= target) hi = mid; else lo = mid + 1;
                }
                SER_CHECK(lo <= kb && TM.goff[cl] + lo < TM.cap);
                /* ... and the same lane finishes the column: closed-form pick inside the item's run, new a or b */
                const double rest = SER_SUB(target, lo > k0 ? SER_ADD(base, val[lo - 1]) : base);
                const int c = c0 + cl;
                const uint2 g4 = *reinterpret_cast<const uint2 *>(TM.st4 + 4 * cl);
                SerStep st;
                st.cur = (int)(g4.x & 0xffffu); st.bound = (int)(g4.x >> 16); st.ocur = (int)(g4.y & 0xffffu); st.kb = kb;
                st.nones = TM.gones[cl]; st.N = N; st.rev = step;
                int q, n;
                SerWeights w = wt;
                if constexpr (MANY) { w.A = TM.wcol[4 * cl + 0]; w.g = TM.wcol[4 * cl + 1]; w.inv_g = TM.wcol[4 * cl + 2]; w.hs = TM.wcol[4 * cl + 3]; }
                const double le = SER_SUB(ser_item_eval(w, st, TM.pos + TM.goff[cl], lo, &q, &n), TM.lmax[cl]);
                const int pick = q - n + 1 + ser_run_pick<MANY ? 0 : 1>(w, n, le, 0.0, rest);
                if (step == 0) { changed += pick != sm.a16[c]; sm.a16[c] = (uint16_t)pick; }
                else { changed += (N - pick) != sm.b16[c]; sm.b16[c] = (uint16_t)(N - pick); }
              }
              __syncwarp(); /* the column's lanes (one warp, the same ones in the next pass) see its new boundary */
            }
            /* no team barrier between the steps: the b-step's geometry + maximum pass maps columns to the same lanes */
            PHASE_MARK(4);
          }
        };
        /* Warp batches: the same step for a few consecutive columns served by ONE warp on its own (no CTA barrier; the warps of
         * the CTA drift through their batches independently, so one warp's dependent chains are the other warps' issue slots).
         * A column's lpc lanes each own a contiguous chunk of its items through all passes: log-weights + maximum, then run
         * weights accumulated straight into the chunk's cumulative sums (no item -> column map, no per-column tables: geometry,
         * maximum and uniforms stay in the lanes' registers), scan of the chunk totals, search + pick.  Same arithmetic, item
         * by item and sum by sum, as the group form. */
        auto gibbs_warp = [&](uint16_t *posw, double *valw, double *wcolw, const int lane, const int c0, const int e0, const int nc,
                              const int lsh) {
          constexpr int TAB = MANY ? 0 : 1;
          const int lpc = 1 << lsh, units = nc << lsh, sub = lane & (lpc - 1);
          const bool live = lane < units;
          const int cl = live ? (lane >> lsh) : 0, c = c0 + cl, head = lane & ~(lpc - 1);
          const int off_c = p.off[c] - e0;
          __syncwarp(); /* the previous batch is done with the slices */
          if (live) { /* postings: the lane expands its run of wq words; the prefix table gives its first slot */
            const int wq = (W + lpc - 1) >> lsh, w0 = sub * wq, w1 = min(W, w0 + wq);
            uint32_t vv[8];
#pragma unroll
            for (int k = 0; k < 8; k++) vv[k] = w0 + k < w1 ? V[(w0 + k) * Cs + c] : 0u;
            const int first = w0 < w1 ? ser_pre_at<BG>(V + c, PRE + c, Cs, w0) : 0;
            uint16_t *out = posw + off_c + first;
            for (int wb = w0; wb < w1; wb += 8) {
              if (wb > w0) {
#pragma unroll
                for (int k = 0; k < 8; k++) vv[k] = wb + k < w1 ? V[(wb + k) * Cs + c] : 0u;
              }
#pragma unroll
              for (int k = 0; k < 8; k++) {
                uint32_t v = vv[k];
                while (v) { *out++ = (uint16_t)(32 * (wb + k) + SER_FFS(v) - 1); v &= v - 1u; }
              }
            }
          }
          double u_a = 0.0, u_b = 0.0; /* the column's two uniforms (mcmc.c:951, :963 -> :909): drawn by its first lane */
          SerWeights w = wt;
          if (live && sub == 0) {
            const int taxon = p.order[c];
            if (p.mode == SER_MODE_REPLAY) {
              const long long u0 = sc.cursor + (MANY ? 6 * (long long)M : 6) + 2 * taxon;
              u_a = tape[u0]; u_b = tape[u0 + 1];
            } else {
              uint32_t o[4];
              ser_philox4x32_10((uint32_t)taxon, SER_BLK_AB, sc.sweep, 0u, p.seed, gchain, o);
              u_a = ser_u53(o[0], o[1]); u_b = ser_u53(o[2], o[3]);
            }
            if constexpr (MANY) { /* the column's own weights */
              SerWeights wo;
              big_col_weights(cd4, p.Mpad, c, &wo);
              ser_set_weights_own(&wo, wo.c, wo.cc, wo.d, wo.dd, N);
              wcolw[4 * cl + 0] = wo.A; wcolw[4 * cl + 1] = wo.g; wcolw[4 * cl + 2] = wo.inv_g; wcolw[4 * cl + 3] = wo.hs;
            }
          }
          u_a = __shfl_sync(0xffffffffu, u_a, head); u_b = __shfl_sync(0xffffffffu, u_b, head);
          __syncwarp(); /* postings (and the columns' weights) are visible to the column's lanes */
          if constexpr (MANY) { w.A = wcolw[4 * cl + 0]; w.g = wcolw[4 * cl + 1]; w.inv_g = wcolw[4 * cl + 2]; w.hs = wcolw[4 * cl + 3]; }
          const uint16_t *pos = posw + off_c;
          double *val = valw + off_c;
#pragma unroll 1
          for (int step = 0; step < 2; step++) {
            const SerStep st = step == 0 ? ser_step_a<BG>(V + c, PRE + c, Cs, W, N, sm.a16[c], sm.b16[c])
                                         : ser_step_b<BG>(V + c, PRE + c, Cs, W, N, sm.a16[c], sm.b16[c]);
            const int kb = st.kb, chunk = (kb + lpc) >> lsh;
            const int k0 = live ? min(kb + 1, sub * chunk) : 0, k1 = live ? min(kb + 1, k0 + chunk) : 0;
            const int qfirst = (k0 > 0 && k0 < k1) ? ser_item_q(st, pos, k0 - 1) : -1; /* last candidate of the item before the chunk */
            double lm = -1.0e300;
            for (int kk = k0; kk < k1; kk++) { /* log-weights of the chunk's items (ser_item_eval), their maximum */
              const int q = kk < kb ? ser_item_q(st, pos, kk) : st.bound;
              const double L = ser_fma(ser_i2d(kk - st.ocur), w.A, SER_MUL(ser_i2d(q - st.cur), w.g));
              val[kk] = L;
              lm = ser_fmax(lm, L);
            }
            for (int o = lpc >> 1; o > 0; o >>= 1) lm = ser_fmax(lm, __shfl_xor_sync(0xffffffffu, lm, o));
            double tot = 0.0;
            int qprev = qfirst;
            for (int kk = k0; kk < k1; kk++) { /* log-weight -> run weight -> cumulative weight inside the chunk */
              const int q = kk < kb ? ser_item_q(st, pos, kk) : st.bound;
              tot = SER_ADD(tot, ser_item_weight_cached<TAB>(w, val[kk], q - qprev, lm));
              val[kk] = tot;
              qprev = q;
            }
            double incl = tot; /* inclusive scan of the chunk totals over the column's lanes */
            for (int o = 1; o < lpc; o <<= 1) {
              const double tt = __shfl_up_sync(0xffffffffu, incl, o);
              if (sub >= o) incl = SER_ADD(incl, tt);
            }
            const double total = __shfl_sync(0xffffffffu, incl, lane | (lpc - 1));
            const double before = __shfl_up_sync(0xffffffffu, incl, 1);
            const double base = sub ? before : 0.0, target = SER_MUL(step ? u_b : u_a, total);
            if (k0 < k1 && incl >= target && (sub == 0 || base < target)) { /* the first chunk that reaches the target */
              int lo = k0, hi = k1 - 1;
              while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (SER_ADD(base, val[mid]) >= target) hi = mid; else lo = mid + 1;
              }
              SER_CHECK(lo <= kb && off_c + lo < p.big_wcap);
              /* ... and the same lane finishes the column: closed-form pick inside the item's run, new a or b */
              const double rest = SER_SUB(target, lo > k0 ? SER_ADD(base, val[lo - 1]) : base);
              int q, n;
              const double le = SER_SUB(ser_item_eval(w, st, pos, lo, &q, &n), lm);
              const int pick = q - n + 1 + ser_run_pick<TAB>(w, n, le, 0.0, rest);
              if (step == 0) { changed += pick != sm.a16[c]; sm.a16[c] = (uint16_t)pick; }
              else { changed += (N - pick) != sm.b16[c]; sm.b16[c] = (uint16_t)(N - pick); }
            }
            __syncwarp(); /* the column's lanes see its new boundary; the chunk sums are consumed */
          }
        };
        if constexpr (WB) {
          /* column batches, one warp each, claimed from a shared-memory counter (the widest columns first) */
          const int warp = tid >> 5, lane = tid & 31;
          uint16_t *posw = sm.pos + (size_t)warp * p.big_wcap;
          double *valw = sm.val + (size_t)warp * p.big_wcap, *wcolw = sm.wcol + (MANY ? 128 * warp : 0);
          __syncthreads(); /* publishes H and this sweep's weights; the batch counter is zero (reset behind the last barrier) */
          PHASE_MARK(0);
          for (;;) {
            int bt = 0;
            if (lane == 0) bt = atomicAdd(sm.bctr, 1);
            bt = __shfl_sync(0xffffffffu, bt, 0);
            if (bt >= p.big_nb) break;
            const int4 bd = __ldg(p.bbat + bt);
            gibbs_warp(posw, valw, wcolw, lane, bd.x, bd.z, bd.y & 0xffff, bd.y >> 16);
          }
          PHASE_MARK(3); /* warp 0's batches; what follows up to the barrier is its wait for the last batch of the CTA */
        } else {
          BigTeam TM;
          TM.pos = sm.pos; TM.val = sm.val; TM.cap = p.big_icap; TM.goff = sm.goff; TM.gones = sm.gones; TM.lmax = sm.lmax;
          TM.st4 = sm.st4; TM.uab = sm.uab; TM.wcol = sm.wcol;
#pragma unroll 1
          for (int g = 0; g < p.big_ng; g++) {
            const int c0 = p.bgrp[2 * g], e0 = p.bgrp[2 * g + 1], c1 = p.bgrp[2 * g + 2], e1 = p.bgrp[2 * g + 3], nc = c1 - c0;
            int lpc = 1, lsh = 0;
            while (lpc < 8 && nc * lpc * 2 <= C) { lpc <<= 1; lsh++; }
            gibbs_team(TM, tid, C, c0, e0, c1, e1, lsh);
          }
        }
        __syncthreads();
        PHASE_MARK(4);
        if (WB && tid == 0) *sm.bctr = 0; /* every warp has left the batch loop; the next sweep's loop starts behind several barriers */
        const bool exact = sampling && s == p.sweeps_per_call - 1;
        {
          int t1 = 0, len = 0, T1, LEN, CH;
          double tsum = 0.0;
          for (int c = tid; c < M; c += C) {
            const int t1c = ser_col_popc<BG>(V + c, PRE + c, Cs, sm.a16[c], sm.b16[c]), lenc = sm.b16[c] - sm.a16[c];
            t1 += t1c; len += lenc;
            if (MANY || exact) { /* mcmc_logl's per-taxon term, mcmc.c:643-644 */
              const int f1 = p.ones[c] - t1c, f0 = lenc - t1c, t0 = N - lenc - f1;
              SerWeights w = wt;
              if constexpr (MANY) big_col_weights(cd4, p.Mpad, c, &w);
              const double term = SER_ADD(SER_ADD(SER_ADD(SER_MUL((double)t0, w.cc), SER_MUL((double)f0, w.d)), SER_MUL((double)t1c, w.dd)),
                                          SER_MUL((double)f1, w.c));
              tsum += term;
              if (exact) TERMS[p.order[c]] = term;
            }
          }
          if constexpr (MANY) {
            double ll;
            block_sum3d(t1, len, changed, tsum, sm.red, sm.redd, ps.buf, &T1, &LEN, &CH, &ll);
            sc.t1a = T1; sc.f1a = (int)p.ones_total - T1; sc.f0a = LEN - T1; sc.t0a = N * M - LEN - sc.f1a;
            sc.loglik = ll;
          } else {
            block_sum3(t1, len, changed, sm.red, ps.buf, &T1, &LEN, &CH);
            totals_from(p, wt, T1, LEN, &sc.t0a, &sc.f0a, &sc.t1a, &sc.f1a, &sc.loglik);
          }
          sc.counters[2] += CH;
          if (exact) {
            if (tid < 32) {
              double acc = 0.0;
              for (int m = 0; m < M; m++) acc = SER_ADD(acc, TERMS[m]);
              if (tid == 0) sm.draws_cd[7] = acc;
            }
            __syncthreads();
            sc.loglik = sm.draws_cd[7];
          }
        }

        /* ================= 16 proposals for pi ================= */
        ps.k = 0;
        for (int prop = 0; prop < 16; prop++) {
          const int kind = prop == 0 ? 3 : ((prop - 1) % 3);
          PHASE_MARK(prop == 0 ? 5 : prop == 1 ? 11 : 8 + (prop - 2) % 3); /* the time since the last mark was the previous proposal's */
          int dt0 = 0, dt1 = 0, nz = 0, D0, D1;
          double delta, tsum = 0.0;
          auto add = [&](int c, int x0, int x1) { /* a column's deltas into the thread's partial sums */
            dt0 += x0; dt1 += x1; nz |= (x0 | x1) != 0;
            if constexpr (MANY) if (x0 | x1) { SerWeights w; big_col_weights(cd4, p.Mpad, c, &w); tsum += ser_term(w, x0, x1); }
          };
          if (kind == 0) { /* pi1 */
            const int i = ser_draw_int(sm.draws_pi[ps.k], N);
            int j = ser_draw_int(sm.draws_pi[ps.k + 1], N - 1);
            ps.k += 2;
            if (j >= i) j++;
            const int lo = min(i, j), hi = max(i, j);
            if (ser_is_hard(hd, i) && ser_hard_count(hd, lo, hi) > 1) continue;
            auto redo = [&](int c, int *x0, int *x1) { ser_pi1_delta(V + c, Cs, sm.a16[c], sm.b16[c], i, j, x0, x1); };
            for (int c = tid; c < M; c += C) { int x0, x1; redo(c, &x0, &x1); add(c, x0, x1); }
            if (!mh_decide_big<MANY>(p, sm, wt, cd4, ps, TERMS, dt0, dt1, nz, tsum, exact, &D0, &D1, &delta, redo)) continue;
            PHASE_MARK(8);
            for (int c = tid; c <= M; c += C) {
              if (c < M) {
                int a = sm.a16[c], b = sm.b16[c]; ser_pi1_apply_ab(&a, &b, i, j); sm.a16[c] = (uint16_t)a; sm.b16[c] = (uint16_t)b;
                ser_col_rotate<BG>(V + c, Cs, W, i, j, PRE + c);
              } else ser_col_rotate(sm.hcol, 1, W, i, j, sm.hpre);
            }
            for (int n = lo + tid; n <= hi; n += C) sm.tmp16[n] = sm.rpi[i < j ? (n < j ? n + 1 : i) : (n > j ? n - 1 : i)];
            __syncthreads();
            for (int n = lo + tid; n <= hi; n += C) sm.rpi[n] = sm.tmp16[n];
            big_rebuild_hard(sm, N);
            PHASE_MARK(12);
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
            auto redo = [&](int c, int *x0, int *x1) { ser_pi2_delta<BG>(V + c, PRE + c, Cs, sm.a16[c], sm.b16[c], i, j, inc1, inc2, x0, x1); };
            for (int c = tid; c < M; c += C) { int x0, x1; redo(c, &x0, &x1); add(c, x0, x1); }
            if (!mh_decide_big<MANY>(p, sm, wt, cd4, ps, TERMS, dt0, dt1, nz, tsum, exact, &D0, &D1, &delta, redo)) continue;
            for (int c = tid; c <= M; c += C) {
              if (c < M) {
                int a = sm.a16[c], b = sm.b16[c];
                const int ain = ser_in_window(a, i, j + 1, inc1, inc2), bin = ser_in_window(b, i, j + 1, inc1, inc2);
                ser_mirror_ab(a, b, ain, bin, i + j + 1, &a, &b);
                sm.a16[c] = (uint16_t)a; sm.b16[c] = (uint16_t)b;
              }
              if (c < M) ser_col_reverse<BG>(V + c, Cs, W, i, j, PRE + c);
              else ser_col_reverse(sm.hcol, 1, W, i, j, sm.hpre);
            }
            for (int n = i + tid; n <= j; n += C) sm.tmp16[n] = sm.rpi[i + j - n];
            __syncthreads();
            for (int n = i + tid; n <= j; n += C) sm.rpi[n] = sm.tmp16[n];
            big_rebuild_hard(sm, N);
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
            auto redo = [&](int c, int *x0, int *x1) {
              if (hb) ser_pi3_delta<true, BG>(V + c, PRE + c, Cs, hd, g, sm.a16[c], sm.b16[c], inc1, inc2, x0, x1, __ldg(p.hbits + c));
              else ser_pi3_delta<false, BG>(V + c, PRE + c, Cs, hd, g, sm.a16[c], sm.b16[c], inc1, inc2, x0, x1);
            };
            for (int c = tid; c < M; c += C) { int x0, x1; redo(c, &x0, &x1); add(c, x0, x1); }
            if (!mh_decide_big<MANY>(p, sm, wt, cd4, ps, TERMS, dt0, dt1, nz, tsum, exact, &D0, &D1, &delta, redo)) continue;
            PHASE_MARK(10);
            for (int n = g.i + tid; n <= g.j; n += C) sm.perm16[n] = (uint16_t)ser_pi3_perm(hd, g, n);
            __syncthreads();
            for (int c = tid; c < M; c += C) {
              int a = sm.a16[c], b = sm.b16[c];
              const int ain = ser_in_window(a, g.i, g.j + 1, inc1, inc2), bin = ser_in_window(b, g.i, g.j + 1, inc1, inc2);
              ser_mirror_ab(a, b, ain, bin, g.i + g.j + 1, &a, &b);
              sm.a16[c] = (uint16_t)a; sm.b16[c] = (uint16_t)b;
              ser_col_permute<BG>(V + c, Cs, W, g.i, g.j, sm.perm16, PRE + c);
            }
            for (int n = g.i + tid; n <= g.j; n += C) sm.tmp16[n] = sm.rpi[sm.perm16[n]];
            __syncthreads();
            for (int n = g.i + tid; n <= g.j; n += C) sm.rpi[n] = sm.tmp16[n];
            PHASE_MARK(13);
            sc.counters[6]++;
          }
          sc.t0a += D0; sc.f0a -= D0; sc.t1a += D1; sc.f1a -= D1;
          sc.loglik = SER_ADD(sc.loglik, delta);
          __syncthreads();
        }

        if (p.mode == SER_MODE_REPLAY) sc.cursor += (MANY ? 8 * (long long)M : 6 + 2 * (long long)M) + ps.k;
        else sc.sweep++;
        sc.counters[7]++;
        PHASE_MARK(10); /* the 16th proposal is a pi3 */
      }
      if (sc.flags & 1) break;

      if (sampling) {
        const int sidx = sc.n_samples - p.sample_base;
        if (sidx < p.max_samples) {
          const size_t row = (size_t)chain * p.max_samples + sidx;
          if (p.store >= SER_STORE_PI)
            for (int pos = tid; pos < N; pos += C) p.samp_pi[row * N + sm.rpi[pos]] = (uint16_t)pos;
          if constexpr (MANY) { sc.c = sm.draws_cd[0]; sc.d = sm.draws_cd[1]; } /* taxon 0's c, d (compute_exp_data, mcmc.c:56-57) */
          if (p.store >= SER_STORE_FULL) {
            for (int c = tid; c < M; c += C) {
              p.samp_a[row * M + p.order[c]] = sm.a16[c]; p.samp_b[row * M + p.order[c]] = sm.b16[c];
              if constexpr (MANY) { p.samp_cd_all[(row * 2 + 0) * M + p.order[c]] = cd4[c]; p.samp_cd_all[(row * 2 + 1) * M + p.order[c]] = cd4[2 * p.Mpad + c]; }
            }
            if (tid == 0) { p.samp_cdl[row * 3 + 0] = sc.c; p.samp_cdl[row * 3 + 1] = sc.d; p.samp_cdl[row * 3 + 2] = sc.loglik; }
          }
        }
        if constexpr (MANY) { sc.c = sm.draws_cd[0]; sc.d = sm.draws_cd[1]; }
        sc.sum_negll = SER_ADD(sc.sum_negll, -sc.loglik);
        sc.sum_ec = SER_ADD(sc.sum_ec, exp(sc.c));
        sc.sum_ed = SER_ADD(sc.sum_ed, exp(sc.d));
        sc.n_samples++;
      }
    }

    __syncthreads();
    for (int c = tid; c < M; c += C) {
      p.ab[(size_t)chain * 2 * p.Mpad + c] = sm.a16[c];
      p.ab[(size_t)chain * 2 * p.Mpad + p.Mpad + c] = sm.b16[c];
    }
    for (int n = tid; n < N; n += C) p.rpi[(size_t)chain * p.Npad + n] = sm.rpi[n];
    if (tid == 0) {
      if constexpr (MANY) { /* the scalar slots carry taxon 0's c, d */
        sc.c = cd4[p.col0]; sc.cc = cd4[p.Mpad + p.col0]; sc.d = cd4[2 * p.Mpad + p.col0]; sc.dd = cd4[3 * p.Mpad + p.col0];
      }
      p.scal[chain] = sc;
    }
  }
}
