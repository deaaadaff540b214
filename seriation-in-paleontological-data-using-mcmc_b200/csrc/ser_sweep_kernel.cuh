/* ser_sweep_kernel.cuh -- the sweep kernel: one CTA per chain, one thread per taxon column (scalar and per-taxon c, d).
 * Part of the single translation unit ser_kernels.cu (included there, in this order). */

/* ------------------------------------------------------------------ the sweep kernel */
struct PropState { /* thread-uniform bookkeeping of the pi part */
  int k;           /* next slot of draws_pi */
  int buf;         /* reduction double-buffer index */
};

/* sum of the M per-taxon terms in taxon order (the reference's own order of additions).  One warp walks
 * the dependent chain and publishes the result; the others wait at the barrier instead of issuing the same
 * M additions (the kernel is issue-bound and shares the SM with other chains).  terms[] is published. */
__device__ __forceinline__ double sequential_term_sum(const Smem &sm, int M)
{
  if (threadIdx.x < 32) {
    double acc = 0.0;
    for (int m = 0; m < M; m++) acc = SER_ADD(acc, sm.terms[m]);
    if (threadIdx.x == 0) sm.draws_cd[7] = acc;
  }
  __syncthreads();
  return sm.draws_cd[7];
}

/* block sum of three ints and one double behind one barrier (per-taxon c, d) */
__device__ __forceinline__ void block_sum3d(int v0, int v1, int v2, double x, int *red, double *redd, int &buf, int *o0, int *o1,
                                            int *o2, double *ox)
{
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
  v0 = __reduce_add_sync(0xffffffffu, v0);
  v1 = __reduce_add_sync(0xffffffffu, v1);
  v2 = __reduce_add_sync(0xffffffffu, v2);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  int *r = red + buf * (SER_MAX_WARPS * 4);
  double *rd = redd + buf * SER_MAX_WARPS;
  if (lane == 0) { r[warp * 4 + 0] = v0; r[warp * 4 + 1] = v1; r[warp * 4 + 2] = v2; rd[warp] = x; }
  __syncthreads();
  int s0 = 0, s1 = 0, s2 = 0;
  double sx = 0.0;
  if (lane < nwarp) { s0 = r[lane * 4 + 0]; s1 = r[lane * 4 + 1]; s2 = r[lane * 4 + 2]; sx = rd[lane]; }
  s0 = __reduce_add_sync(0xffffffffu, s0);
  s1 = __reduce_add_sync(0xffffffffu, s1);
  s2 = __reduce_add_sync(0xffffffffu, s2);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sx += __shfl_xor_sync(0xffffffffu, sx, o);
  buf ^= 1;
  *o0 = s0; *o1 = s1; *o2 = s2; *ox = sx;
}

/* MH tail shared by the three proposals (mcmc.c:1261/:1441/:1636): block-reduce the integer deltas, form
 * delta, accept.  Every thread computes the same decision.
 * Scalar c, d: delta follows from the integer totals; if they cancel while single taxa changed, the
 * reference's sequential float sum (mcmc.c:1214/1435/1630) may leave a residual whose SIGN decides whether
 * a draw is consumed, so that sum is re-created exactly.
 * Per-taxon c, d (MANY): delta is a float sum over taxa -- reduced in parallel (good to ~1e-12), re-done in the
 * reference's order when the sign could be ambiguous.  On a sampled sweep every accepted delta is the
 * reference's own sum, so the saved log-likelihood carries its bits. */
template <bool MANY>
__device__ __forceinline__ bool mh_decide(const KParams &p, const Smem &sm, const SerWeights &wt, PropState &ps, int taxon,
                                          bool is_taxon, int dt0, int dt1, bool exact, int *D0, int *D1, double *delta_out)
{
  int nz;
  double delta;
  bool seq = false;
  auto reference_sum = [&]() { /* per-taxon terms in the reference's operand order, added in taxon order */
    double acc = 0.0;
    __syncthreads(); /* terms[] may still be read from an earlier call */
    if (is_taxon) sm.terms[taxon] = ser_term(wt, dt0, dt1);
    __syncthreads();
    acc = sequential_term_sum(sm, p.M);
    return acc;
  };
  if constexpr (MANY) {
    block_sum3d(dt0, dt1, (dt0 | dt1) != 0, is_taxon ? ser_term(wt, dt0, dt1) : 0.0, sm.red, sm.redd, ps.buf, D0, D1, &nz, &delta);
    if (!nz) delta = 0.0;
    else if (fabs(delta) < 1e-7) { delta = reference_sum(); seq = true; }
  } else {
    block_sum3(dt0, dt1, (dt0 | dt1) != 0, sm.red, ps.buf, D0, D1, &nz);
    if (*D0 == 0 && *D1 == 0) {
      delta = 0.0;
      if (nz) { delta = reference_sum(); seq = true; }
    } else {
      delta = ser_term(wt, *D0, *D1);
    }
  }
  bool accept = delta >= 0.0;
  if (!accept) accept = delta > sm.logdraw[ps.k++];
  if (accept && exact && !seq && nz) delta = reference_sum();
  *delta_out = delta;
  return accept;
}

#define SER_UNIT_MAXL 32 /* most lanes that serve one column (a whole warp) */
/* A unit of the Gibbs phase: `lpc` = 1 << lsh adjacent lanes serve column c, this lane is number `sub` of them;
 * off = first item of the column (KParams::unit_tab, built by ser_run_create) */
struct Unit {
  int c, sub, lsh, lpc, off;
  bool live;
};
__device__ __forceinline__ Unit unit_load(const KParams &p, int u, int n_units)
{
  Unit un;
  un.live = u < n_units;
  const uint2 t = un.live ? __ldg(p.unit_tab + u) : make_uint2(0u, 0u);
  un.c = (int)(t.x & 0xffffu); un.sub = (int)((t.x >> 16) & 0xffu); un.lsh = (int)(t.x >> 24); un.lpc = 1 << un.lsh;
  un.off = (int)t.y;
  return un;
}
/* the step geometry the column's owner published */
__device__ __forceinline__ SerStep unit_step(const Smem &sm, int c, int N, int step)
{
  const uint2 g4 = *reinterpret_cast<const uint2 *>(sm.st4 + 4 * c); /* cur, bound | ocur, kb */
  SerStep it;
  it.cur = (int)(g4.x & 0xffffu); it.bound = (int)(g4.x >> 16); it.ocur = (int)(g4.y & 0xffffu); it.kb = (int)(g4.y >> 16);
  it.nones = sm.ones16[c]; it.N = N; it.rev = step;
  return it;
}

/* MAXT = largest block the instantiation is launched with: the small-block instantiation may use
 * more registers per thread (shared memory, not registers, limits residency there).
 * MANY = per-taxon c, d (manycd = 1, mcmc.c:777-785, :807-815): same choreography; the Beta draws, weights
 * and likelihood terms are per thread, the geometric run sums are evaluated on the fly (no shared table)
 * and delta / loglik are float sums over taxa (mh_decide). */
template <int MAXT, int MINB, bool MANY>
__global__ void __launch_bounds__(MAXT, MINB) ser_sweep_kernel(KParams p)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem sm;
  smem_layout(&sm, smem_raw, p.N, p.W, p.C, p.I, MANY ? 1 : 0, p.Ival);

  const int tid = threadIdx.x, N = p.N, M = p.M, C = p.C, W = p.W;
  uint32_t *col = sm.V + tid;
  uint16_t *pre = sm.pre + tid;
  const bool is_taxon = tid < M, is_col = tid <= M;
  __shared__ unsigned int s_item, s_gchain;

  /* static per column (the same for every chain this CTA serves) */
  int taxon = 0, off_c = 0, ones_c = 0;
  uint32_t hbits_c = 0u; /* bit k: this column has a one at the k-th hard site (static; nh <= 32) */
  if (is_taxon) {
    taxon = p.order[tid]; /* the taxon this column holds: indexes the tape, the samples, terms[] */
    off_c = p.off[tid];
    ones_c = p.ones[tid];
    sm.ones16[tid] = (uint16_t)ones_c;
    hbits_c = p.hbits[tid];
  }

  /* ---- persistent grid: the CTAs pull (chain, chunk of calls) work items from a queue until it is empty.
   * Items are numbered chunk-major, so a chain's chunks are claimed in order; a chunk waits until the chain's
   * previous chunk has published its state (done[chain], release / acquire).  The holder of an earlier item is
   * always a running CTA, so the wait cannot deadlock, whatever the grid size. */
  for (;;) {
  __syncthreads(); /* the previous item is done with shared memory (and with s_item) */
  if (tid == 0) s_item = atomicAdd(p.queue, 1u);
  __syncthreads();
  const unsigned int item = s_item;
  if (item >= p.n_items) break;
  const int chunk = (int)(item / (unsigned int)p.n_chains), chain = (int)(item - (unsigned int)chunk * (unsigned int)p.n_chains);
  const int call_lo = chunk * p.chunk_calls, call_hi = min(p.n_calls, call_lo + p.chunk_calls);
  if (chunk > 0) {
    if (tid == 0) {
      const volatile unsigned int *dn = p.done + chain;
      while ((int)(*dn - (p.chunk_base + (unsigned int)chunk)) < 0) __nanosleep(64);
      __threadfence();
    }
    __syncthreads();
  }
  /* the global id lives in shared memory, read at the draws: held in a register across the sweep loop it costs this
   * register-capped kernel 0.5 % (B200, g2s2) */
  if (tid == 0) s_gchain = global_chain(p, chain); /* visible after the barrier below the state loads */
  const unsigned int &gchain = s_gchain;

  /* ---- load chain state (L1-bypassing loads: another SM may have written it a moment ago) */
  ChainScalars sc;
  {
    const int4 *src = reinterpret_cast<const int4 *>(p.scal + chain);
    int4 *dst = reinterpret_cast<int4 *>(&sc);
#pragma unroll
    for (int q = 0; q < (int)(sizeof(ChainScalars) / 16); q++) dst[q] = __ldcg(src + q);
  }
  for (int n = tid; n < N; n += C) sm.rpi[n] = __ldcg(p.rpi + (size_t)chain * p.Npad + n);
  int a = 0, b = 0;
  double c = p.c0, cc = p.cc0, d = p.d0, dd = p.dd0; /* MANY: this taxon's c, log(1-e^c), d, log(1-e^d) */
  if (is_taxon) {
    a = __ldcg(p.ab + (size_t)chain * 2 * p.Mpad + tid);
    b = __ldcg(p.ab + (size_t)chain * 2 * p.Mpad + p.Mpad + tid);
    if constexpr (MANY) {
      const double *cd = p.cd4 + (size_t)chain * 4 * p.Mpad + tid;
      c = __ldcg(cd); cc = __ldcg(cd + p.Mpad); d = __ldcg(cd + 2 * p.Mpad); dd = __ldcg(cd + 3 * p.Mpad);
    }
  }
  __syncthreads();
  if (sc.flags & SER_FLAG_COLUMNS) { /* the bit columns travel with the chain between work items */
    const uint32_t *gv = p.gVc + (size_t)chain * W * C + tid;
    for (int w = 0; w < W; w++) sm.V[w * C + tid] = __ldcg(gv + (size_t)w * C);
    ser_col_build_pre(sm.V + tid, sm.pre + tid, C, W);
  } else {
    build_columns(p, sm);
  }
  __syncthreads();
  rebuild_hard(p, sm);
  __syncthreads();

  bool pos_dirty = true; /* the postings of this chain are not in shared memory yet */
  const double *tape = nullptr;
  long long tape_len = 0;
  if (p.mode == SER_MODE_REPLAY) {
    tape = p.tape + p.tape_off[chain];
    tape_len = (long long)(p.tape_off[chain + 1] - p.tape_off[chain]);
  }

  SerWeights wt;
  if constexpr (MANY) {
    ser_set_weights_own(&wt, c, cc, d, dd, N);
  } else {
    wt.H = sm.H;
    wt.hmax = 0;
    set_weights(wt, sc.c, sc.cc, sc.d, sc.dd);
  }
  wt.eps = p.eps;
  SerHard hd;
  hd.hcol = sm.V + M; hd.hpre = sm.pre + M; hd.hp = sm.hp; hd.C = C; hd.W = W; hd.N = N; hd.nh = p.nh; hd.rank_tab = sm.hrank; hd.nonhard_tab = sm.nhpos;
  PropState ps;
  ps.k = 0; ps.buf = 0;

  for (int call = call_lo; call < call_hi && !(sc.flags & 1); call++) {
    const bool sampling = call >= p.burn_calls; /* burn-in calls first, then sampling calls (mcmc.c:140-143, :180-185) */
    for (int s = 0; s < p.sweeps_per_call; s++) {
      __syncthreads(); /* every thread is done reading the previous sweep's staged draws */
      PHASE_T0();
      double ua = 0.0, ub = 0.0;
      if constexpr (MANY) {
        /* ================= draws: M Betas for c, M for d, 2M uniforms, then the pi draws ================= */
        double yc = 0.0, lyc = 0.0, l1c = 0.0, yd = 0.0, lyd = 0.0, l1d = 0.0;
        if (p.mode == SER_MODE_REPLAY) {
          const long long need = sc.cursor + 8 * (long long)M;
          if (need > tape_len) { sc.flags |= 1; break; }
          for (int t = tid; t < SER_PI_DRAWS; t += C) {
            const long long idx = need + t;
            const double u = idx < tape_len ? tape[idx] : 0.5;
            sm.draws_pi[t] = u;
            sm.logdraw[t] = log(u);
          }
          if (is_taxon) {
            const double *tc = tape + sc.cursor + 3 * taxon, *td = tape + sc.cursor + 3 * (long long)M + 3 * taxon;
            yc = tc[0]; lyc = tc[1]; l1c = tc[2];
            yd = td[0]; lyd = td[1]; l1d = td[2];
            ua = tape[sc.cursor + 6 * (long long)M + 2 * taxon]; ub = tape[sc.cursor + 6 * (long long)M + 2 * taxon + 1];
          }
        } else {
          for (int t = tid; t < SER_PI_DRAWS; t += C) {
            const double u = ser_stream_uniform(p.seed, gchain, sc.sweep, SER_BLK_PI, (uint32_t)t);
            sm.draws_pi[t] = u;
            sm.logdraw[t] = log(ser_pos(u));
          }
          if (is_taxon) { /* Beta(1+f1_m, 1+t0_m) and Beta(1+f0_m, 1+t1_m) from the taxon's own counts */
            const int t1 = ser_col_popc(col, pre, C, a, b), len = b - a;
            const int f1 = ones_c - t1, f0 = len - t1, t0 = N - len - f1;
            const uint32_t blk = SER_BLK_MANYCD + 4u * (uint32_t)taxon;
            yc = ser_beta_from_gammas(ser_gamma_ge1(1.0 + (double)f1, p.seed, gchain, sc.sweep, blk),
                                      ser_gamma_ge1(1.0 + (double)t0, p.seed, gchain, sc.sweep, blk + 1u));
            yd = ser_beta_from_gammas(ser_gamma_ge1(1.0 + (double)f0, p.seed, gchain, sc.sweep, blk + 2u),
                                      ser_gamma_ge1(1.0 + (double)t1, p.seed, gchain, sc.sweep, blk + 3u));
            if (yc > 0.0) { lyc = ser_log(yc); l1c = ser_log(SER_SUB(1.0, ser_exp(lyc))); }
            if (yd > 0.0) { lyd = ser_log(yd); l1d = ser_log(SER_SUB(1.0, ser_exp(lyd))); }
            uint32_t o[4];
            ser_philox4x32_10((uint32_t)taxon, SER_BLK_AB, sc.sweep, 0u, p.seed, gchain, o);
            ua = ser_u53(o[0], o[1]); ub = ser_u53(o[2], o[3]);
          }
        }
        /* ================= c_m, d_m (mcmc_samplebeta per taxon) ================= */
        if (is_taxon) {
          if (yc > 0.0 && SER_MINC <= lyc && lyc <= SER_MAXC) { c = lyc; cc = l1c; }
          if (yd > 0.0 && SER_MIND <= lyd && lyd <= SER_MAXD) { d = lyd; dd = l1d; }
          ser_set_weights_own(&wt, c, cc, d, dd, N);
          sm.wcol[4 * tid + 0] = wt.A; sm.wcol[4 * tid + 1] = wt.g; sm.wcol[4 * tid + 2] = wt.inv_g; sm.wcol[4 * tid + 3] = wt.hs;
          if (taxon == 0) { sm.draws_cd[0] = c; sm.draws_cd[1] = d; }
        }
        sc.counters[0] += M; sc.counters[1] += M;

      } else {
        /* ================= stage this sweep's draws ================= */
        if (p.mode == SER_MODE_REPLAY) {
          const long long need = sc.cursor + 6 + 2 * (long long)M;
          if (need > tape_len) { sc.flags |= 1; break; } /* uniform across the CTA */
          if (tid < 6) sm.draws_cd[tid] = tape[sc.cursor + tid];
          for (int t = tid; t < SER_PI_DRAWS; t += C) {
            const long long idx = need + t;
            const double u = idx < tape_len ? tape[idx] : 0.5;
            sm.draws_pi[t] = u;
            sm.logdraw[t] = log(u);
          }
          if (is_taxon) { ua = tape[sc.cursor + 6 + 2 * taxon]; ub = tape[sc.cursor + 7 + 2 * taxon]; }
        } else {
          if (tid < 4) { /* Beta(1+f1a,1+t0a) and Beta(1+f0a,1+t1a) as Gamma ratios (mcmc.c:790, :820) */
            const int cnt = tid == 0 ? sc.f1a : tid == 1 ? sc.t0a : tid == 2 ? sc.f0a : sc.t1a;
            const double g = ser_gamma_ge1(1.0 + (double)cnt, p.seed, gchain, sc.sweep, (uint32_t)tid);
            const double go = __shfl_xor_sync(0xfu, g, 1);
            if (tid == 0 || tid == 2) {
              const double y = ser_beta_from_gammas(g, go);
              double val = tid == 0 ? sc.c : sc.d, l1m = tid == 0 ? sc.cc : sc.dd;
              const double lo = tid == 0 ? SER_MINC : SER_MIND, hi = tid == 0 ? SER_MAXC : SER_MAXD;
              if (y > 0.0) { /* mcmc_samplebeta, mcmc.c:751-765 */
                const double ly = ser_log(y);
                if (lo <= ly && ly <= hi) { val = ly; l1m = ser_log(SER_SUB(1.0, ser_exp(ly))); }
              }
              sm.draws_cd[tid] = val; sm.draws_cd[tid + 1] = l1m;
            }
          }
          for (int t = tid; t < SER_PI_DRAWS; t += C) {
            const double u = ser_stream_uniform(p.seed, gchain, sc.sweep, SER_BLK_PI, (uint32_t)t);
            sm.draws_pi[t] = u;
            sm.logdraw[t] = log(ser_pos(u));
          }
          if (is_taxon) {
            uint32_t o[4];
            ser_philox4x32_10((uint32_t)taxon, SER_BLK_AB, sc.sweep, 0u, p.seed, gchain, o);
            ua = ser_u53(o[0], o[1]); ub = ser_u53(o[2], o[3]);
          }
        }
        __syncthreads();

        /* ================= c and d (mcmc_samplec / mcmc_sampled) ================= */
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
        /* geometric partial sums for this sweep's g (shared by all taxa: c, d are scalar) */
        wt.hmax = min(ser_hmax(wt.g, N), SER_HCAP - 1);
        for (int m = tid; m <= wt.hmax; m += C) sm.H[m] = ser_h_entry(wt.g, m);
        __syncthreads();

      }

      /* ================= a/b Gibbs (mcmc_sampleab, mcmc.c:918-996) =================
       * item formulation (ser_chain_core.h): postings of the column, then for the a-step and
       * the b-step, per column group: per-column maximum + cached log-weights (units), item weights
       * (dense over the CTA), per-column scan + item search (units), pick inside the run (owner). */
      PHASE_MARK(8);
      /* The per-column loops of this phase -- postings, maximum, cumulative weights -- are served by UNITS: a column
       * with many ones gets 2, 4, .. 32 adjacent lanes (static table, built per column group from the columns' item
       * counts), so the longest serial loop of a pass is a few items (g2s2: 95 items in the heaviest column).  With one
       * thread per column the warp that owns the 32 heaviest columns was the critical path of every pass while the
       * other nine waited at the barrier (30 % of the sweep's cycles). */
      /* The postings survive from sweep to sweep: an accepted adjacent swap or site move patches them in place (below);
       * only a segment reversal or a pi3 move (1 % of the proposals each) marks them for this rebuild. */
      if (pos_dirty)
      for (int ub = 0; ub < p.n_units; ub += C) { /* postings: lane `sub` expands its share of the column's words */
        const Unit un = unit_load(p, ub + tid, p.n_units);
        if (un.live) {
          const int wq = (W + un.lpc - 1) >> un.lsh, w0 = un.sub * wq, w1 = min(W, w0 + wq);
          if (w0 < w1) {
            uint16_t *out = sm.pos + un.off + sm.pre[w0 * C + un.c]; /* the prefix table gives the first slot */
            for (int w = w0; w < w1; w++) {
              uint32_t v = sm.V[w * C + un.c];
              while (v) { *out++ = (uint16_t)(32 * w + SER_FFS(v) - 1); v &= v - 1u; }
            }
            SER_CHECK(out <= sm.pos + un.off + (int)sm.ones16[un.c] && un.off + (int)sm.ones16[un.c] <= p.I);
          }
        }
      }
      pos_dirty = false;
      PHASE_MARK(9);
      int changed = 0;
#pragma unroll 1
      for (int step = 0; step < 2; step++) {
        if (is_taxon) { /* step geometry of the own column and its uniform, published for the units */
          sm.terms[tid] = step == 0 ? ua : ub; /* terms[] is idle during the Gibbs phase */
          const SerStep st = step == 0 ? ser_step_a(col, pre, C, W, N, a, b) : ser_step_b(col, pre, C, W, N, a, b);
          *reinterpret_cast<uint2 *>(sm.st4 + 4 * tid) =
              make_uint2((uint32_t)st.cur | ((uint32_t)st.bound << 16), (uint32_t)st.ocur | ((uint32_t)st.kb << 16));
        }
        __syncthreads(); /* also: the postings are complete */
        PHASE_MARK(10);
#pragma unroll 1
        for (int g = 0; g < p.n_groups; g++) { /* columns grp_c[g]..grp_c[g+1] = items grp_e[g]..grp_e[g+1] = units grp_u[g]..grp_u[g+1] */
          const int e0 = p.grp_e[g], e1 = p.grp_e[g + 1], ug1 = p.grp_u[g + 1];
          if (g) __syncthreads(); /* the previous group's scans are done with val */
          /* maximum log-weight per column (the reference's z, mcmc.c:727-730).  The lanes also leave every item's
           * log-weight in val[] and its run length in ncache[], so that the dense pass below needs neither the step
           * geometry nor the postings. */
          for (int ub = p.grp_u[g]; ub < ug1; ub += C) {
            const Unit un = unit_load(p, ub + tid, ug1);
            double lm = -1.0e300;
            if (un.live) {
              const SerStep it = unit_step(sm, un.c, N, step);
              const uint16_t *pos = sm.pos + un.off;
              SerWeights w = wt;
              if constexpr (MANY) { w.A = sm.wcol[4 * un.c + 0]; w.g = sm.wcol[4 * un.c + 1]; }
              double *Lc = sm.val + (un.off - e0);
              uint16_t *nc = sm.ncache + (un.off - e0);
              SER_CHECK(un.off - e0 >= 0 && un.off - e0 + it.kb <= p.Ival);
              for (int kk = un.sub; kk <= it.kb; kk += un.lpc) {
                int q, n;
                const double L = ser_item_eval(w, it, pos, kk, &q, &n);
                Lc[kk] = L; nc[kk] = (uint16_t)n;
                lm = ser_fmax(lm, L);
              }
            }
#pragma unroll
            for (int o = 1; o < SER_UNIT_MAXL; o <<= 1) {
              const double t = __shfl_xor_sync(0xffffffffu, lm, o);
              if (o < un.lpc) lm = ser_fmax(lm, t);
            }
            if (un.live && un.sub == 0) sm.lmax[un.c] = lm;
          }
          __syncthreads();
          PHASE_MARK(19);
          {
            uint32_t ck_next = e0 + tid < e1 ? p.item_col[e0 + tid] : 0u; /* item -> column map, fetched one iteration ahead */
            for (int e = e0 + tid; e < e1; e += C) { /* log-weight -> run weight, in place */
              const uint32_t ck = ck_next;
              if (e + C < e1) ck_next = p.item_col[e + C];
              const int c = (int)(ck >> 16), kk = (int)(ck & 0xffffu);
              if (kk <= (int)sm.st4[4 * c + 3]) { /* inside the step's bound */
                SER_CHECK(e - e0 >= 0 && e - e0 <= p.Ival && c < M);
                int m; double ye;
                if constexpr (MANY) { /* the column's own weights; geometric sums on the fly */
                  SerWeights w;
                  w.g = sm.wcol[4 * c + 1]; w.inv_g = sm.wcol[4 * c + 2]; w.hs = sm.wcol[4 * c + 3];
                  w.eps = p.eps; w.H = nullptr; w.hmax = N + 1;
                  sm.val[e - e0] = ser_run_sum<0>(w, (int)sm.ncache[e - e0], SER_SUB(sm.val[e - e0], sm.lmax[c]), &m, &ye);
                } else {
                  sm.val[e - e0] = ser_run_sum<1>(wt, (int)sm.ncache[e - e0], SER_SUB(sm.val[e - e0], sm.lmax[c]), &m, &ye);
                }
#if defined(SER_PHASE_TIMING) && defined(SER_COUNT_ITEMS) /* how many items are evaluated / lie above the LOGEPSILON floor */
                atomicAdd(&ser_phase_cycles[20], 1ull); if (m) atomicAdd(&ser_phase_cycles[21], 1ull);
#endif
              }
            }
          }
          __syncthreads();
          PHASE_MARK(11);
          /* cumulative weights and the item the uniform falls into (mcmc_randompick, mcmc.c:901-915).  Lane `sub` owns
           * the contiguous chunk [k0, k1) of the column's items: serial sums inside the chunk (chunk-relative), a scan of
           * the chunk totals over the column's lanes; the lane whose chunk is the first to reach target = U x total
           * finds the item inside its chunk and leaves (item, target - weight before the item) for the owner. */
          for (int ub = p.grp_u[g]; ub < ug1; ub += C) { /* warp-uniform trip count: the shuffles need every lane */
            const Unit un = unit_load(p, ub + tid, ug1);
            const int kb = un.live ? (int)sm.st4[4 * un.c + 3] : 0;
            const double u01 = un.live ? sm.terms[un.c] : 0.0;
            double *val = sm.val + (un.off - e0);
            const int chunk = (kb + un.lpc) >> un.lsh, k0 = min(kb + 1, un.sub * chunk), k1 = min(kb + 1, k0 + chunk);
            SER_CHECK(!un.live || (un.off - e0 >= 0 && un.off - e0 + k1 <= p.Ival + 1 && un.c >= p.grp_c[g] && un.c < p.grp_c[g + 1]));
            double tot = 0.0;
            if (un.live) for (int kk = k0; kk < k1; kk++) { tot = SER_ADD(tot, val[kk]); val[kk] = tot; }
            double incl = tot; /* inclusive scan of the chunk totals over the column's lanes */
#pragma unroll
            for (int o = 1; o < SER_UNIT_MAXL; o <<= 1) {
              const double t = __shfl_up_sync(0xffffffffu, incl, o);
              if (o < un.lpc && un.sub >= o) incl = SER_ADD(incl, t);
            }
            const int lane = tid & 31;
            const double total = __shfl_sync(0xffffffffu, incl, (lane | (un.lpc - 1)));
            const double before = __shfl_up_sync(0xffffffffu, incl, 1);
            const double base = un.sub ? before : 0.0, target = SER_MUL(u01, total);
            if (un.live && k0 < k1 && incl >= target && (un.sub == 0 || base < target)) {
              int lo = k0, hi = k1 - 1; /* first item of the chunk whose cumulative weight reaches the target */
              while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (SER_ADD(base, val[mid]) >= target) hi = mid; else lo = mid + 1;
              }
              sm.pick16[un.c] = (uint16_t)lo;
              sm.terms[un.c] = SER_SUB(target, lo > k0 ? SER_ADD(base, val[lo - 1]) : base);
            }
          }
          PHASE_MARK(12);
        }
        __syncthreads();
        if (is_taxon) { /* the owner: closed-form pick inside the item's run */
          const SerStep st = unit_step(sm, tid, N, step);
          SER_CHECK((int)sm.pick16[tid] <= st.kb);
          int q, n;
          const double le = SER_SUB(ser_item_eval(wt, st, sm.pos + off_c, (int)sm.pick16[tid], &q, &n), sm.lmax[tid]);
          const int pick = q - n + 1 + ser_run_pick<MANY ? 0 : 1>(wt, n, le, 0.0, sm.terms[tid]);
          if (step == 0) { changed += pick != a; a = pick; }
          else { changed += (N - pick) != b; b = N - pick; }
        }
        PHASE_MARK(18);
      }
      /* the log-likelihood is only ever observed after the last sweep of a sampling call
       * (mcmc_save_chain); there it is formed with the reference's own sequential sums */
      const bool exact = sampling && s == p.sweeps_per_call - 1;
      if constexpr (MANY) {
        {
          int t1 = 0, len = 0, T1, LEN, CH;
          double term = 0.0, ll;
          if (is_taxon) {
            t1 = ser_col_popc(col, pre, C, a, b); len = b - a;
            const int f1 = ones_c - t1, f0 = len - t1, t0 = N - len - f1;
            term = SER_ADD(SER_ADD(SER_ADD(SER_MUL((double)t0, wt.cc), SER_MUL((double)f0, wt.d)), SER_MUL((double)t1, wt.dd)),
                           SER_MUL((double)f1, wt.c));
          }
          block_sum3d(t1, len, changed, term, sm.red, sm.redd, ps.buf, &T1, &LEN, &CH, &ll);
          sc.t1a = T1; sc.f1a = (int)p.ones_total - T1; sc.f0a = LEN - T1; sc.t0a = N * M - LEN - sc.f1a;
          sc.loglik = ll;
          sc.counters[2] += CH;
          if (exact) { /* mcmc_logl's own order */
            if (is_taxon) sm.terms[taxon] = term;
            __syncthreads();
            sc.loglik = sequential_term_sum(sm, M);
          }
        }
      } else {
        int t1 = 0, len = 0;
        if (is_taxon) { t1 = ser_col_popc(col, pre, C, a, b); len = b - a; }
        {
          int T1, LEN, CH;
          block_sum3(t1, len, changed, sm.red, ps.buf, &T1, &LEN, &CH);
          totals_from(p, wt, T1, LEN, &sc.t0a, &sc.f0a, &sc.t1a, &sc.f1a, &sc.loglik);
          sc.counters[2] += CH;
          if (exact) { /* mcmc_logl, mcmc.c:625-648: sum over taxa of t0*cc + f0*d + t1*dd + f1*c */
            if (is_taxon) {
              const int f1 = ones_c - t1, f0 = len - t1, t0 = N - len - f1;
              sm.terms[taxon] = SER_ADD(SER_ADD(SER_ADD(SER_MUL((double)t0, wt.cc), SER_MUL((double)f0, wt.d)), SER_MUL((double)t1, wt.dd)),
                                        SER_MUL((double)f1, wt.c));
            }
            __syncthreads();
            sc.loglik = sequential_term_sum(sm, M);
          }
        }
      }

      /* ================= 16 proposals for pi (mcmc.c:237-243) ================= */
      ps.k = 0;
      PHASE_MARK(13);
      for (int prop = 0; prop < 16; prop++) {
        PHASE_MARK(14 + (prop <= 1 ? 3 : ((prop + 1) % 3))); /* charged to the PREVIOUS proposal's kind: 14 pi1, 15 pi2, 16 pi3, 17 swap */
        /* order: pi2(swap), then 5 x (pi1, pi2(0), pi3) */
        const int kind = prop == 0 ? 3 : ((prop - 1) % 3); /* 0 pi1, 1 pi2(0), 2 pi3, 3 pi2(swap) */
        int dt0 = 0, dt1 = 0, D0, D1;
        double delta;
        if (kind == 0) { /* ---------------- mcmc_samplepi1, mcmc.c:1127-1308 */
          const int i = ser_draw_int(sm.draws_pi[ps.k], N);
          int j = ser_draw_int(sm.draws_pi[ps.k + 1], N - 1);
          ps.k += 2;
          if (j >= i) j++;
          const int lo = min(i, j), hi = max(i, j);
          const int nhw = ser_hard_count(hd, lo, hi); /* hard sites in the window */
          if (ser_is_hard(hd, i) && nhw > 1) continue;
          if (is_taxon) ser_pi1_delta(col, C, a, b, i, j, &dt0, &dt1);
          if (!mh_decide<MANY>(p, sm, wt, ps, taxon, is_taxon, dt0, dt1, exact, &D0, &D1, &delta)) continue;
          if (is_taxon) ser_pi1_apply_ab(&a, &b, i, j);
          if (is_taxon && !pos_dirty) { /* the column's postings inside the window: shifted by one, the moved site's one goes to the other end */
            uint16_t *pc = sm.pos + off_c;
            const int k0 = ser_rank1(col, pre, C, lo), k1 = ser_rank1(col, pre, C, hi + 1); /* on the column BEFORE the move */
            const int moved = ser_col_bit(col, C, i);
            if (i < j) {
              for (int k = k0 + moved; k < k1; k++) pc[k - moved] = (uint16_t)(pc[k] - 1);
              if (moved) pc[k1 - 1] = (uint16_t)j;
            } else {
              for (int k = k1 - 1 - moved; k >= k0; k--) pc[k + moved] = (uint16_t)(pc[k] + 1);
              if (moved) pc[k0] = (uint16_t)j;
            }
          }
          if (is_col) ser_col_rotate(col, C, W, i, j, pre);
          for (int n = lo + tid; n <= hi; n += C)
            sm.tmp16[n] = sm.rpi[i < j ? (n < j ? n + 1 : i) : (n > j ? n - 1 : i)];
          __syncthreads();
          for (int n = lo + tid; n <= hi; n += C) sm.rpi[n] = sm.tmp16[n];
          if (nhw) { __syncthreads(); rebuild_hard(p, sm); } /* the hard column only changed if the window holds a hard site */
          sc.counters[3]++;
        } else if (kind == 1 || kind == 3) { /* ---------------- mcmc_samplepi2, mcmc.c:1311-1486 */
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
          const int nhw = ser_hard_count(hd, i, j);
          if (nhw > 1) continue;
          const int inc1 = ser_draw_int(sm.draws_pi[ps.k], 2), inc2 = ser_draw_int(sm.draws_pi[ps.k + 1], 2);
          ps.k += 2;
          if (is_taxon) ser_pi2_delta(col, pre, C, a, b, i, j, inc1, inc2, &dt0, &dt1);
          if (!mh_decide<MANY>(p, sm, wt, ps, taxon, is_taxon, dt0, dt1, exact, &D0, &D1, &delta)) continue;
          if (is_taxon) {
            const int ain = ser_in_window(a, i, j + 1, inc1, inc2), bin = ser_in_window(b, i, j + 1, inc1, inc2);
            ser_mirror_ab(a, b, ain, bin, i + j + 1, &a, &b);
          }
          if (kind == 3) { /* adjacent swap: at most one posting of the column changes, between i and i + 1 */
            if (is_taxon && !pos_dirty) {
              const int b0 = ser_col_bit(col, C, i), b1 = ser_col_bit(col, C, j);
              if (b0 != b1) sm.pos[off_c + ser_rank1(col, pre, C, i)] = (uint16_t)(b0 ? j : i);
            }
          } else pos_dirty = true;
          if (is_col) ser_col_reverse(col, C, W, i, j, pre);
          for (int n = i + tid; 2 * n < i + j; n += C) { /* mirror the site order: disjoint pairs, no staging */
            const uint16_t t = sm.rpi[n];
            sm.rpi[n] = sm.rpi[i + j - n]; sm.rpi[i + j - n] = t;
          }
          if (nhw) { __syncthreads(); rebuild_hard(p, sm); }
          sc.counters[kind == 1 ? 4 : 5]++;
        } else { /* ---------------- mcmc_samplepi3, mcmc.c:1489-1682 */
          const int nfree = N - p.nh;
          if (nfree < 2) continue;
          const int r1 = ser_draw_int(sm.draws_pi[ps.k], nfree), r2 = ser_draw_int(sm.draws_pi[ps.k + 1], nfree - 1);
          ps.k += 2;
          int ir, jr;
          if (r1 <= r2) { ir = r1; jr = r2 + 1; } else { ir = r2; jr = r1; }
          const SerPi3 g = ser_pi3_window(hd, ir, jr);
          const int inc1 = ser_draw_int(sm.draws_pi[ps.k], 2), inc2 = ser_draw_int(sm.draws_pi[ps.k + 1], 2);
          ps.k += 2;
          if (is_taxon) {
            if (p.nh <= 32) ser_pi3_delta<true>(col, pre, C, hd, g, a, b, inc1, inc2, &dt0, &dt1, hbits_c);
            else ser_pi3_delta<false>(col, pre, C, hd, g, a, b, inc1, inc2, &dt0, &dt1);
          }
          if (!mh_decide<MANY>(p, sm, wt, ps, taxon, is_taxon, dt0, dt1, exact, &D0, &D1, &delta)) continue;
          for (int n = g.i + tid; n <= g.j; n += C) sm.perm16[n] = (uint16_t)ser_pi3_perm(hd, g, n);
          __syncthreads();
          if (is_taxon) {
            const int ain = ser_in_window(a, g.i, g.j + 1, inc1, inc2), bin = ser_in_window(b, g.i, g.j + 1, inc1, inc2);
            ser_mirror_ab(a, b, ain, bin, g.i + g.j + 1, &a, &b);
            ser_col_permute(col, C, W, g.i, g.j, sm.perm16, pre);
          }
          for (int n = g.i + tid; n <= g.j; n += C) { /* the permutation is an involution: disjoint pairs */
            const int m2 = sm.perm16[n];
            if (m2 > n) { const uint16_t t = sm.rpi[n]; sm.rpi[n] = sm.rpi[m2]; sm.rpi[m2] = t; }
          }
          pos_dirty = true;
          sc.counters[6]++;
        }
        /* accepted: fold the integer deltas into the totals (the reference recounts, mcmc.c:1303) */
        sc.t0a += D0; sc.f0a -= D0; sc.t1a += D1; sc.f1a -= D1;
        sc.loglik = SER_ADD(sc.loglik, delta);
        SER_CHECK(ps.k <= SER_PI_DRAWS && a >= 0 && a <= b && b <= N);
        __syncthreads(); /* columns / hard mask / rpi visible before the next proposal */
      }

      PHASE_MARK(16);
      if (p.mode == SER_MODE_REPLAY) sc.cursor += (MANY ? 8 * (long long)M : 6 + 2 * (long long)M) + ps.k;
      else sc.sweep++;
      sc.counters[7]++;
    }
    if (sc.flags & 1) break;

    /* ================= thinned sample (mcmc_save_chain + compute_exp_data) ================= */
    if constexpr (MANY) {
      if (sampling) {
        const int sidx = sc.n_samples - p.sample_base;
        const double c_first = sm.draws_cd[0], d_first = sm.draws_cd[1]; /* taxon 0's c, d (compute_exp_data, mcmc.c:56-57) */
        if (sidx < p.max_samples) {
          const size_t row = (size_t)chain * p.max_samples + sidx;
          if (p.store >= SER_STORE_PI)
            for (int pos = tid; pos < N; pos += C) p.samp_pi[row * N + sm.rpi[pos]] = (uint16_t)pos;
          if (p.store >= SER_STORE_FULL) {
            if (is_taxon) {
              p.samp_a[row * M + taxon] = (uint16_t)a; p.samp_b[row * M + taxon] = (uint16_t)b;
              p.samp_cd_all[(row * 2 + 0) * M + taxon] = c; p.samp_cd_all[(row * 2 + 1) * M + taxon] = d;
            }
            if (tid == 0) { p.samp_cdl[row * 3 + 0] = c_first; p.samp_cdl[row * 3 + 1] = d_first; p.samp_cdl[row * 3 + 2] = sc.loglik; }
          }
        }
        sc.c = c_first; sc.d = d_first;
        sc.sum_negll = SER_ADD(sc.sum_negll, -sc.loglik);
        sc.sum_ec = SER_ADD(sc.sum_ec, exp(c_first));
        sc.sum_ed = SER_ADD(sc.sum_ed, exp(d_first));
        sc.n_samples++;
      }
    } else {
      if (sampling) {
        const int sidx = sc.n_samples - p.sample_base;
        if (sidx < p.max_samples) {
          const size_t row = (size_t)chain * p.max_samples + sidx;
          if (p.store >= SER_STORE_PI)
            for (int pos = tid; pos < N; pos += C) p.samp_pi[row * N + sm.rpi[pos]] = (uint16_t)pos;
          if (p.store >= SER_STORE_FULL) {
            if (is_taxon) { p.samp_a[row * M + taxon] = (uint16_t)a; p.samp_b[row * M + taxon] = (uint16_t)b; }
            if (tid == 0) { p.samp_cdl[row * 3 + 0] = sc.c; p.samp_cdl[row * 3 + 1] = sc.d; p.samp_cdl[row * 3 + 2] = sc.loglik; }
          }
        }
        sc.sum_negll = SER_ADD(sc.sum_negll, -sc.loglik);
        sc.sum_ec = SER_ADD(sc.sum_ec, exp(sc.c));
        sc.sum_ed = SER_ADD(sc.sum_ed, exp(sc.d));
        sc.n_samples++;
      }
    }
  }

  /* ---- save chain state (incl. the bit columns) and publish the item */
  __syncthreads();
  sc.flags |= SER_FLAG_COLUMNS;
  {
    uint32_t *gv = p.gVc + (size_t)chain * W * C + tid;
    for (int w = 0; w < W; w++) gv[(size_t)w * C] = sm.V[w * C + tid];
  }
  if (is_taxon) {
    p.ab[(size_t)chain * 2 * p.Mpad + tid] = (uint16_t)a;
    p.ab[(size_t)chain * 2 * p.Mpad + p.Mpad + tid] = (uint16_t)b;
  }
  for (int n = tid; n < N; n += C) p.rpi[(size_t)chain * p.Npad + n] = sm.rpi[n];
  if constexpr (MANY) {
    if (is_taxon) {
      double *cd = p.cd4 + (size_t)chain * 4 * p.Mpad + tid;
      cd[0] = c; cd[p.Mpad] = cc; cd[2 * p.Mpad] = d; cd[3 * p.Mpad] = dd;
      if (taxon == 0) { sm.draws_cd[0] = c; sm.draws_cd[1] = cc; sm.draws_cd[2] = d; sm.draws_cd[3] = dd; }
    }
    __syncthreads();
    if (tid == 0) { sc.c = sm.draws_cd[0]; sc.cc = sm.draws_cd[1]; sc.d = sm.draws_cd[2]; sc.dd = sm.draws_cd[3]; } /* the scalar slots carry taxon 0's c, d */
  }
  if (tid == 0) p.scal[chain] = sc;
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    *(volatile unsigned int *)(p.done + chain) = p.chunk_base + (unsigned int)chunk + 1u;
  }
  } /* work items */
}

