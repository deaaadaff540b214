/* ser_aux_kernels.cuh -- export / consistency-check kernels, the cross-chain kernels (stats, selection, pair order, posterior sums, alive counts) and the peak micro-benchmarks.
 * Part of the single translation unit ser_kernels.cu (included there, in this order). */

/* ------------------------------------------------------------------ export / check kernels */
/* int32 view of one chain's state incl. the derived per-taxon counts (mcmc_count01) */
__global__ void ser_export_kernel(KParams p, int chain, int *out_a, int *out_b, int *out_pi, int *out_rpi, int *out_cnt)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  AuxSmem sm;
  aux_layout(&sm, smem_raw, p.N);
  const int tid = threadIdx.x, C = blockDim.x;
  for (int n = tid; n < p.N; n += C) sm.rpi[n] = p.rpi[(size_t)chain * p.Npad + n];
  __syncthreads();
  for (int n = tid; n < p.N; n += C) { out_rpi[n] = sm.rpi[n]; out_pi[sm.rpi[n]] = n; }
  for (int c = tid; c < p.M; c += C) {
    const int a = p.ab[(size_t)chain * 2 * p.Mpad + c], b = p.ab[(size_t)chain * 2 * p.Mpad + p.Mpad + c];
    const int t1 = taxon_count(p, sm.rpi, c, a, b), ones = p.ones[c];
    const int tx = p.order[c];
    out_a[tx] = a; out_b[tx] = b;
    out_cnt[tx] = p.N - (b - a) - (ones - t1); out_cnt[p.M + tx] = (b - a) - t1;
    out_cnt[2 * p.M + tx] = t1; out_cnt[3 * p.M + tx] = ones - t1;
  }
}

/* mcmc_consistent (mcmc.c:999-1094) for every chain; flags |= 2 a/b range, 4 permutation,
 * 8 hard-site order, 16 totals / log-likelihood */
__global__ void ser_check_kernel(KParams p, int *bad_count)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  AuxSmem sm;
  aux_layout(&sm, smem_raw, p.N);
  const int chain = blockIdx.x, tid = threadIdx.x, C = blockDim.x, N = p.N, M = p.M;
  __shared__ int s_flags;
  if (tid == 0) s_flags = 0;
  for (int n = tid; n < N; n += C) { sm.rpi[n] = p.rpi[(size_t)chain * p.Npad + n]; sm.tmp16[n] = 0xffff; }
  __syncthreads();
  for (int n = tid; n < N; n += C) {
    const int site = sm.rpi[n];
    if (site >= N) { atomicOr(&s_flags, 4); sm.rpi[n] = 0; }
    else sm.tmp16[site] = (uint16_t)n; /* pi */
  }
  __syncthreads();
  for (int n = tid; n < N; n += C) if (sm.tmp16[n] == 0xffff) atomicOr(&s_flags, 4);
  if (tid == 0) { /* hard sites in increasing position in file order */
    int last = -1, cnt = 0;
    for (int n = 0; n < N; n++)
      if (p.hard[n]) { cnt++; if (last >= 0 && (int)sm.tmp16[n] < last) s_flags |= 8; last = sm.tmp16[n]; }
    if (cnt != p.nh) atomicOr(&s_flags, 8);
  }
  int t1 = 0, len = 0;
  double llp = 0.0; /* manycd: the log-likelihood is a sum of per-taxon terms */
  for (int c = tid; c < M; c += C) {
    const int a = p.ab[(size_t)chain * 2 * p.Mpad + c], b = p.ab[(size_t)chain * 2 * p.Mpad + p.Mpad + c];
    if (!(0 <= a && a <= b && b <= N)) atomicOr(&s_flags, 2);
    else {
      const int k1 = taxon_count(p, sm.rpi, c, a, b);
      t1 += k1; len += b - a;
      if (p.manycd) {
        const double *cd = p.cd4 + (size_t)chain * 4 * p.Mpad + c;
        const int f1 = p.ones[c] - k1, f0 = (b - a) - k1, t0 = N - (b - a) - f1;
        llp += (double)t0 * cd[p.Mpad] + (double)f0 * cd[2 * p.Mpad] + (double)k1 * cd[3 * p.Mpad] + (double)f1 * cd[0];
      }
    }
  }
  int buf = 0, T1, LEN, dummy;
  block_sum3(t1, len, 0, sm.red, buf, &T1, &LEN, &dummy);
  __shared__ double s_ll[32];
  if (p.manycd) {
    for (int o = 16; o > 0; o >>= 1) llp += __shfl_xor_sync(0xffffffffu, llp, o);
    if ((tid & 31) == 0) s_ll[tid >> 5] = llp;
    __syncthreads();
  }
  if (tid == 0) {
    const ChainScalars sc = p.scal[chain];
    SerWeights wt;
    set_weights(wt, sc.c, sc.cc, sc.d, sc.dd);
    int t0a, f0a, t1a, f1a;
    double ll;
    totals_from(p, wt, T1, LEN, &t0a, &f0a, &t1a, &f1a, &ll);
    if (p.manycd) { ll = 0.0; for (int w = 0; w < (C + 31) / 32; w++) ll += s_ll[w]; }
    /* the reference allows 1e-8 absolute (mcmc.c:1084); on large matrices |loglik| ~ 1e6 and the taxon-order
     * sum of a sampled sweep differs from this recount's closed form by more than that in the last bits */
    if (t0a != sc.t0a || f0a != sc.f0a || t1a != sc.t1a || f1a != sc.f1a || fabs(ll - sc.loglik) > 1e-8 + 1e-12 * fabs(ll)) s_flags |= 16;
    const int fl = s_flags | (sc.flags & 1);
    if (fl) atomicAdd(bad_count, 1);
    p.scal[chain].flags = (sc.flags & (1 | SER_FLAG_COLUMNS)) | fl;
  }
}

/* ------------------------------------------------------------------ cross-chain kernels */
/* Destinations of a cross-chain kernel: the same buffer on this device and, for the single-process multi-GPU
 * path (ser_multi.cuh), on every peer device -- the kernel's stores ARE the all-gather (NVLink peer stores). */
#define SER_MAX_PEERS 8
struct PeerPtrs {
  void *p[SER_MAX_PEERS];
  int n;
};

/* E[-logL] of every local chain (compute_exp_data / print_exp_data, mcmc.c:53-67, divided by the samples taken),
 * written at dst[offset + chain] of every destination */
__global__ void ser_stats_kernel(const ChainScalars *scal, int n, PeerPtrs dst, int offset)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double v = scal[i].n_samples > 0 ? scal[i].sum_negll / (double)scal[i].n_samples : 0.0;
  for (int q = 0; q < dst.n; q++) ((double *)dst.p[q])[offset + i] = v;
}

__device__ double block_reduce_d(double v, double *sh, int op) /* 0 sum, 1 min */
{
  for (int o = 16; o > 0; o >>= 1) {
    const double t = __shfl_xor_sync(0xffffffffu, v, o);
    v = op ? fmin(v, t) : v + t;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  if (lane == 0) sh[warp] = v;
  __syncthreads();
  double r = sh[0];
  for (int w = 1; w < nw; w++) r = op ? fmin(r, sh[w]) : r + sh[w];
  return r;
}

/* choose_chains (script.py:70-99) on one CTA: min, population sigma over all chains, the k
 * smallest inside (min-sigma, min+sigma), ids ascending */
__global__ void ser_select_kernel(const double *e, int n, int k, int *chosen, double *info)
{
  __shared__ double sh[32];
  __shared__ double s_best;
  __shared__ int s_besti;
  const int tid = threadIdx.x, nt = blockDim.x;
  double s = 0.0, mn = 1.0e300;
  for (int i = tid; i < n; i += nt) { s += e[i]; mn = fmin(mn, e[i]); }
  const double mean = block_reduce_d(s, sh, 0) / (double)n;
  mn = block_reduce_d(mn, sh, 1);
  double v = 0.0;
  for (int i = tid; i < n; i += nt) { const double d = e[i] - mean; v += d * d; }
  const double sigma = sqrt(block_reduce_d(v, sh, 0) / (double)n);
  const double lo = mn - sigma, hi = mn + sigma;
  /* k rounds of arg-min over the not-yet-taken candidates, ties by lower id */
  double last_v = -1.0e300;
  int last_i = -1, found = 0;
  for (int r = 0; r < k; r++) {
    double bv = 1.0e300;
    int bi = -1;
    for (int i = tid; i < n; i += nt) {
      const double x = e[i];
      if (!(x > lo && x < hi)) continue;
      if (x < last_v || (x == last_v && i <= last_i)) continue;
      if (x < bv || (x == bv && i < bi)) { bv = x; bi = i; }
    }
    for (int o = 16; o > 0; o >>= 1) {
      const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (oi >= 0 && (bi < 0 || ov < bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
    }
    __syncthreads();
    if (tid == 0) { s_best = 1.0e300; s_besti = -1; }
    __syncthreads();
    for (int w = 0; w < (nt >> 5); w++) {
      if ((tid >> 5) == w && (tid & 31) == 0 && bi >= 0)
        if (s_besti < 0 || bv < s_best || (bv == s_best && bi < s_besti)) { s_best = bv; s_besti = bi; }
      __syncthreads();
    }
    if (s_besti < 0) break;
    last_v = s_best; last_i = s_besti;
    if (tid == 0) chosen[found] = s_besti;
    found++;
    __syncthreads();
  }
  __syncthreads();
  if (tid == 0) {
    for (int r = found; r < k; r++) chosen[r] = -1;
    for (int x = 1; x < found; x++) { /* ids ascending (script.py:98) */
      const int key = chosen[x];
      int y = x - 1;
      while (y >= 0 && chosen[y] > key) { chosen[y + 1] = chosen[y]; y--; }
      chosen[y + 1] = key;
    }
    info[0] = (double)found; info[1] = mn; info[2] = sigma;
  }
}

/* samples of a chain that the store holds */
__device__ __forceinline__ int stored_samples(const ChainScalars *scal, int local, int max_samples)
{
  const int n = scal[local].n_samples;
  return n < max_samples ? n : max_samples;
}

/* Local index of GLOBAL chain g on a run whose local chain c is id_base + c (ids == nullptr), or ids[c] (subset runs,
 * ser_run_create_chains: a handful of chosen chains, so a scan); -1 when the run does not hold g. */
__device__ __forceinline__ int local_chain(int g, int id_base, int n_local, const int *ids)
{
  if (!ids) return (g >= id_base && g < id_base + n_local) ? g - id_base : -1;
  for (int c = 0; c < n_local; c++)
    if (ids[c] == g) return c;
  return -1;
}

/* rows [0, T) of a chain's store taken since sample_base, at most w (fewer only when its replay tape ran out) */
__device__ __forceinline__ int window_rows(const ChainScalars *scal, int local, int sample_base, int w)
{
  const int n = scal[local].n_samples - sample_base;
  return n < 0 ? 0 : n < w ? n : w;
}

/* Which chain block b of a summary kernel reads, and how many rows of its store:
 *   one-shot (chosen != nullptr): the local chain holding global id chosen[b] (none: the block does nothing), sample_base 0 and
 *     rows = max_samples, i.e. every stored sample (the copy-out kernels of an accumulating run pass rows = INT_MAX: T = every
 *     sample taken since accumulation began);
 *   streaming (chosen == nullptr): local chain b, the rows of the window its last sweep launch of w sampling calls filled
 *     (sample_base, rows = w).
 * The chain's T goes to n_out[b] when n_out is given. */
struct SumSel {
  const int *chosen;
  int id_base, n_local;
  const int *ids;
  int sample_base, rows;
  int *n_out;
};

/* local chain of block b (-1: not held) and its T; `lead` = the one thread of the block's chain that writes n_out */
__device__ __forceinline__ int sel_chain(const SumSel &s, const ChainScalars *scal, int b, bool lead, int *T)
{
  const int local = s.chosen ? local_chain(s.chosen[b], s.id_base, s.n_local, s.ids) : b;
  if (local < 0) return -1;
  *T = window_rows(scal, local, s.sample_base, s.rows);
  if (lead && s.n_out) s.n_out[b] = *T;
  return local;
}

/* pair-order counts of a 32 x 32 tile of (i, j) over rows [0, T) of one chain's samples `pi` ([row][N]): the positions of the
 * tile's 64 sites staged through shared memory 32 samples at a time (coalesced rows).  256 threads; thread (tx, ty) adds
 * #{t : pi_t(i0+ty+8r) < pi_t(j0+tx)} to c[r].  Every thread of the block calls it (barriers inside). */
#define SER_PO_TS 32
__device__ __forceinline__ void po_tile(const uint16_t *pi, int N, int T, int i0, int j0, int c[4])
{
  __shared__ uint16_t si[SER_PO_TS][32], sj[SER_PO_TS][32];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int t0 = 0; t0 < T; t0 += SER_PO_TS) {
    const int nt = min(SER_PO_TS, T - t0);
    __syncthreads();
    for (int q = threadIdx.x; q < nt * 32; q += 256) {
      const int t = q >> 5, x = q & 31;
      si[t][x] = i0 + x < N ? pi[(size_t)(t0 + t) * N + i0 + x] : (uint16_t)0;
      sj[t][x] = j0 + x < N ? pi[(size_t)(t0 + t) * N + j0 + x] : (uint16_t)0;
    }
    __syncthreads();
    for (int t = 0; t < nt; t++) {
      const int pj = sj[t][tx];
#pragma unroll
      for (int r = 0; r < 4; r++) c[r] += (int)si[t][ty + 8 * r] < pj;
    }
  }
}

/* Summary kernels: every one serves both the one-shot getters and the streaming accumulators.  Block b reads the chain and rows
 * sel_chain gives it and writes slab b of its output (out + b * stride: a [k][..] output, or the part of a chain's accumulator record,
 * stride acc_layout().ints); add = 0 stores the slab, add = 1 adds into it.  A chain the run does not hold leaves its slab untouched. */

/* pair-order counts (script.py:178-189), one 32 x 32 tile per block, slab blockIdx.z into every destination (peer stores: the slabs
 * are disjoint, so no reduction is needed).  Stored: diagonal -T; added: the diagonal stays 0 (a site is never before itself). */
__global__ void __launch_bounds__(256) ser_po_kernel(const uint16_t *samp_pi, const ChainScalars *scal, int N, int max_samples, SumSel sel,
                                                      PeerPtrs dst, size_t stride, int add)
{
  int T;
  const int local = sel_chain(sel, scal, blockIdx.z, blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0, &T);
  if (local < 0) return;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5; /* 32 x 8 threads; thread (tx, ty) owns j = j0+tx, i = i0+ty+8r */
  const int i0 = blockIdx.y * 32, j0 = blockIdx.x * 32;
  int c[4] = {0, 0, 0, 0};
  po_tile(samp_pi + (size_t)local * max_samples * N, N, T, i0, j0, c);
  const int j = j0 + tx;
  if (j >= N) return;
#pragma unroll
  for (int r = 0; r < 4; r++) {
    const int i = i0 + ty + 8 * r;
    if (i >= N) continue;
    const size_t e = (size_t)blockIdx.z * stride + (size_t)i * N + j;
#pragma unroll
    for (int q = 0; q < SER_MAX_PEERS; q++) /* constant indices: a loop to dst.n would copy the destinations to the stack */
      if (q < dst.n) {
        int *d = (int *)dst.p[q] + e;
        *d = add ? *d + c[r] : (i == j ? -T : c[r]);
      }
  }
}

/* posterior sums (script.py:129-152, :230-276), one chain per block: sum_t pi_t into pi_sum, sum_t a_t / b_t into a_sum / b_sum when
 * given; corr_num[b] = sum_i i * (this block's sum_t pi_t(i)) when given (the one-shot getter) */
__global__ void ser_posterior_kernel(const uint16_t *samp_pi, const uint16_t *samp_a, const uint16_t *samp_b, const ChainScalars *scal,
                                     int N, int M, int max_samples, SumSel sel, int *pi_sum, size_t pi_stride, int *a_sum, int *b_sum,
                                     size_t ab_stride, long long *corr_num, int add)
{
  __shared__ unsigned long long s_corr;
  int T;
  const int local = sel_chain(sel, scal, blockIdx.x, threadIdx.x == 0, &T);
  if (local < 0) return;
  if (threadIdx.x == 0) s_corr = 0;
  const size_t base = (size_t)local * max_samples;
  int *ps = pi_sum + blockIdx.x * pi_stride;
  long long s = 0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    int acc = 0;
    for (int t = 0; t < T; t++) acc += samp_pi[(base + t) * N + i];
    ps[i] = add ? ps[i] + acc : acc;
    s += (long long)i * acc;
  }
  if (a_sum || b_sum)
    for (int m = threadIdx.x; m < M; m += blockDim.x) {
      int sa = 0, sb = 0;
      for (int t = 0; t < T; t++) { sa += samp_a[(base + t) * M + m]; sb += samp_b[(base + t) * M + m]; }
      const size_t e = blockIdx.x * ab_stride + m;
      if (a_sum) a_sum[e] = add ? a_sum[e] + sa : sa;
      if (b_sum) b_sum[e] = add ? b_sum[e] + sb : sb;
    }
  if (!corr_num) return;
  __syncthreads();
  atomicAdd(&s_corr, (unsigned long long)s); /* an integer sum: the same in any order */
  __syncthreads();
  if (threadIdx.x == 0) corr_num[blockIdx.x] = (long long)s_corr;
}

/* alive[j][m] = #{t : a_t(m) <= j <= b_t(m)} (script.py:321-329; closed at b, as the reference tests it).  One thread per taxon: +1 / -1
 * marks at a and b+1 in its own column of the slab.  Stored: the column is zeroed first and the marks are summed down the positions;
 * added: the marks alone go into a difference slab, whose running sum the accumulating getter takes. */
__global__ void ser_alive_kernel(const uint16_t *samp_a, const uint16_t *samp_b, const ChainScalars *scal, int N, int M, int max_samples,
                                 SumSel sel, int *alive, size_t stride, int add)
{
  int T;
  const int local = sel_chain(sel, scal, blockIdx.x, blockIdx.y == 0 && threadIdx.x == 0, &T);
  if (local < 0) return;
  const int m = blockIdx.y * blockDim.x + threadIdx.x;
  if (m >= M) return;
  const size_t base = (size_t)local * max_samples;
  int *col = alive + blockIdx.x * stride + m;
  if (!add)
    for (int j = 0; j < N; j++) col[(size_t)j * M] = 0;
  for (int t = 0; t < T; t++) {
    const int a = samp_a[(base + t) * M + m], b = samp_b[(base + t) * M + m];
    if (a < N) col[(size_t)a * M] += 1;
    if (b + 1 < N) col[(size_t)(b + 1) * M] -= 1;
  }
  if (add) return;
  int acc = 0;
  for (int j = 0; j < N; j++) { acc += col[(size_t)j * M]; col[(size_t)j * M] = acc; }
}

/* taxon pair relations (ser_run_taxon_pairs, DESIGN.md 3.10), one 32 x 32 tile of (m, n) per block, slab blockIdx.z of each output
 * that is not nullptr: first = #{t : a_m < a_n}, last = #{t : b_m < b_n}, precedes = #{t : b_m <= a_n}, coexist = #{t : max(a_m, a_n) <
 * min(b_m, b_n)}.  The tile's 64 taxa are staged 32 samples at a time as (a | b << 16) words from coalesced rows of the a and b stores;
 * thread (tx, ty) owns n = n0 + tx and the four rows m = m0 + 4 ty + r, read as one 16-byte word (a broadcast within the warp).  Its 16
 * counters stay in registers over all T rows: no atomics, so the counts do not depend on the launch shape.  All four are counted
 * whatever is requested: every caller in the project asks for all four, and a one-output variant would be a second kernel (DESIGN.md
 * 3.10). */
__global__ void __launch_bounds__(256) ser_taxon_pair_kernel(const uint16_t *samp_a, const uint16_t *samp_b, const ChainScalars *scal, int M,
                                                             int max_samples, SumSel sel, int *first, int *last, int *precedes, int *coexist,
                                                             size_t stride, int add)
{
  __shared__ __align__(16) uint32_t sm[SER_PO_TS][32], sn[SER_PO_TS][32];
  int T;
  const int local = sel_chain(sel, scal, blockIdx.z, blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0, &T);
  if (local < 0) return;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5, m0 = blockIdx.y * 32, n0 = blockIdx.x * 32;
  const uint16_t *A = samp_a + (size_t)local * max_samples * M, *B = samp_b + (size_t)local * max_samples * M;
  int cf[4] = {0, 0, 0, 0}, cl[4] = {0, 0, 0, 0}, cp[4] = {0, 0, 0, 0}, cc[4] = {0, 0, 0, 0};
  for (int t0 = 0; t0 < T; t0 += SER_PO_TS) {
    const int nt = min(SER_PO_TS, T - t0);
    __syncthreads();
    for (int q = threadIdx.x; q < nt * 32; q += 256) {
      const int t = q >> 5, x = q & 31;
      const size_t row = (size_t)(t0 + t) * M;
      sm[t][x] = m0 + x < M ? (uint32_t)A[row + m0 + x] | (uint32_t)B[row + m0 + x] << 16 : 0u;
      sn[t][x] = n0 + x < M ? (uint32_t)A[row + n0 + x] | (uint32_t)B[row + n0 + x] << 16 : 0u;
    }
    __syncthreads();
    for (int t = 0; t < nt; t++) {
      const uint32_t wn = sn[t][tx];
      const int an = (int)(wn & 0xffffu), bn = (int)(wn >> 16);
      const uint4 w4 = *reinterpret_cast<const uint4 *>(&sm[t][4 * ty]);
      const uint32_t wm[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
      for (int r = 0; r < 4; r++) {
        const int am = (int)(wm[r] & 0xffffu), bm = (int)(wm[r] >> 16);
        cf[r] += am < an;
        cl[r] += bm < bn;
        cp[r] += bm <= an;
        cc[r] += max(am, an) < min(bm, bn);
      }
    }
  }
  const int n = n0 + tx;
  if (n >= M) return;
  int *const outs[4] = {first, last, precedes, coexist};
#pragma unroll
  for (int r = 0; r < 4; r++) {
    const int m = m0 + 4 * ty + r;
    if (m >= M) continue;
    const size_t e = (size_t)blockIdx.z * stride + (size_t)m * M + n;
    const int v[4] = {cf[r], cl[r], cp[r], cc[r]};
#pragma unroll
    for (int q = 0; q < 4; q++)
      if (outs[q]) outs[q][e] = add ? outs[q][e] + v[q] : v[q];
  }
}

/* Error-rate marginals (ser_run_cd_marginals, DESIGN.md 3.11).  Sample t of a chain holds the R rows' c at cd[t * rs + r] and their d
 * at cd[t * rs + d_off + r]: samp_cd_all (rs = 2M, d_off = M) on a manycd run, samp_cdl (rs = 3, d_off = 1, R = 1) on a scalar one.
 * Bin of x on [lo, hi] with s = SER_CD_BINS / (hi - lo): floor((x - lo) * s) rounded step by step, clamped to the bins; x <= lo and
 * NaN give bin 0. */
#define SER_CD_ROWS 32
#define SER_CD_PITCH (SER_CD_BINS + 1) /* a padded shared row: lanes counting the same bin hit 32 different banks */
#define SER_CD_SMEM (2 * SER_CD_ROWS * SER_CD_PITCH * sizeof(int))
__device__ __forceinline__ int cd_bin(double x, double lo, double s)
{
  const double y = __dmul_rn(__dsub_rn(x, lo), s);
  return y >= (double)(SER_CD_BINS - 1) ? SER_CD_BINS - 1 : y > 0.0 ? (int)y : 0;
}

/* One block per (32 rows, chosen chain blockIdx.y); lane = row, so a sample's 32 values are one coalesced load.  Warp 0 folds the
 * rows' exp sums, c_sum / d_sum [R] at slab stride sum_stride: each lane one row, sequentially over t from the stored sum (add) or 0.0,
 * with the sweep kernels' exp and SER_ADD, so the sum is theirs bit for bit.  The other warps stride over the samples and count the
 * rows' c and d bins with shared-memory atomics (integer counts: the same in any order); the block's rows are contiguous in a
 * [R][SER_CD_BINS] slab at stride hist_stride and go out with plain stores.  Both are computed whatever is requested; a nullptr output
 * is not written. */
__global__ void __launch_bounds__(256) ser_cd_hist_kernel(const double *cd, size_t rs, int d_off, int R, const ChainScalars *scal,
                                                          int max_samples, SumSel sel, double *c_sum, double *d_sum, size_t sum_stride,
                                                          int *c_hist, int *d_hist, size_t hist_stride, int add)
{
  extern __shared__ int s_cd[]; /* [2][SER_CD_ROWS][SER_CD_PITCH]: c, then d */
  int T;
  const int local = sel_chain(sel, scal, blockIdx.y, blockIdx.x == 0 && threadIdx.x == 0, &T);
  if (local < 0) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int r0 = blockIdx.x * SER_CD_ROWS, n = min(SER_CD_ROWS, R - r0), r = r0 + lane;
  const double *x = cd + (size_t)local * max_samples * rs + r;
  for (int e = threadIdx.x; e < 2 * SER_CD_ROWS * SER_CD_PITCH; e += blockDim.x) s_cd[e] = 0;
  __syncthreads();
  if (lane < n) {
    if (warp == 0) {
      const size_t e = (size_t)blockIdx.y * sum_stride + r;
      double sc = add && c_sum ? c_sum[e] : 0.0, sd = add && d_sum ? d_sum[e] : 0.0;
      for (int t = 0; t < T; t++) {
        sc = SER_ADD(sc, exp(x[(size_t)t * rs]));
        sd = SER_ADD(sd, exp(x[(size_t)t * rs + d_off]));
      }
      if (c_sum) c_sum[e] = sc;
      if (d_sum) d_sum[e] = sd;
    } else {
      const double sc = (double)SER_CD_BINS / (SER_MAXC - SER_MINC), sd = (double)SER_CD_BINS / (SER_MAXD - SER_MIND);
      int *hc = s_cd + lane * SER_CD_PITCH, *hd = hc + SER_CD_ROWS * SER_CD_PITCH;
      for (int t = warp - 1; t < T; t += nw - 1) {
        atomicAdd(&hc[cd_bin(x[(size_t)t * rs], SER_MINC, sc)], 1);
        atomicAdd(&hd[cd_bin(x[(size_t)t * rs + d_off], SER_MIND, sd)], 1);
      }
    }
  }
  __syncthreads();
  int *const outs[2] = {c_hist, d_hist};
  for (int h = 0; h < 2; h++) {
    if (!outs[h]) continue;
    int *dst = outs[h] + (size_t)blockIdx.y * hist_stride + (size_t)r0 * SER_CD_BINS;
    const int *src = s_cd + h * SER_CD_ROWS * SER_CD_PITCH;
    for (int e = threadIdx.x; e < n * SER_CD_BINS; e += blockDim.x) {
      const int v = src[(e / SER_CD_BINS) * SER_CD_PITCH + e % SER_CD_BINS];
      dst[e] = add ? dst[e] + v : v;
    }
  }
}

/* ------------------------------------------------------------------ convergence diagnostics (ser_run_diagnostics, DESIGN.md 3.7)
 * Quantity q of a chain's stored sample t: 0 = -loglik, 1 = exp(c), 2 = exp(d) (samp_cdl; taxon 0's c, d on a manycd run),
 * 3 + i = pi_t(i), the position of site i.  One block of 32 warps per (chosen chain, 32 consecutive quantities).  The moments
 * read the store with lane = quantity and warp = t mod 32 (coalesced rows), then reduce the 32 partials in warp order.  The
 * autocovariances run one warp per quantity, lane l summing lag k0 + l in t order over centred traces staged 64 samples at a
 * time; a warp stops after the lag block in which a Geyer pair sum turns non-positive.  No sum depends on the grid. */
#define SER_DIAG_TC 64             /* samples per staged chunk */
#define SER_DIAG_SA (SER_DIAG_TC + 1)  /* odd row strides: the staging stores hit distinct banks */
#define SER_DIAG_SB (SER_DIAG_TC + 33)

__device__ __forceinline__ double diag_value(const uint16_t *pi, const double *cdl, int N, int q, int t)
{
  if (q >= 3) return (double)pi[(size_t)t * N + q - 3];
  if (q == 0) return -cdl[(size_t)t * 3 + 2];
  return exp(cdl[(size_t)t * 3 + q - 1]);
}

/* One staged chunk of the lag sums over traces of length len (1024 threads): row j of sA holds val(j, t) for t = t0 .. t0 + 63 and
 * row j of sB for t = t0 + k0 .. t0 + k0 + 95, zero where t >= len or the warp of quantity j has stopped (act[j] == 0).  val(j, t)
 * returns the centred value.  Every thread of the block calls it, between barriers. */
template <class Val>
__device__ __forceinline__ void stage_lag_chunk(double *sA, double *sB, const int *act, int t0, int k0, int len, Val val)
{
  for (int e = threadIdx.x; e < 32 * SER_DIAG_TC; e += 1024) {
    const int t = t0 + (e >> 5), j = e & 31;
    sA[j * SER_DIAG_SA + (e >> 5)] = (act[j] && t < len) ? val(j, t) : 0.0;
  }
  for (int e = threadIdx.x; e < 32 * (SER_DIAG_TC + 32); e += 1024) {
    const int t = t0 + k0 + (e >> 5), j = e & 31;
    sB[j * SER_DIAG_SB + (e >> 5)] = (act[j] && t < len) ? val(j, t) : 0.0;
  }
}

/* warp w's lane l adds the products of its quantity's staged chunk at lag k0 + l, for the chunk's first nt samples, in t order */
__device__ __forceinline__ double lag_chunk_dot(const double *sA, const double *sB, int w, int lane, int nt, double acc)
{
  const double *a = sA + w * SER_DIAG_SA, *b = sB + w * SER_DIAG_SB + lane;
  for (int t = 0; t < nt; t++) acc = fma(a[t], b[t], acc);
  return acc;
}

/* stats [k][3+N][4] = mean, var, ess, lags; halves [k][3+N][4] = mean1, var1, mean2, var2 for quantities [qlo, qhi); n_out[c] = T */
__global__ void __launch_bounds__(1024, 1) ser_diag_kernel(const uint16_t *samp_pi, const double *samp_cdl, const ChainScalars *scal, int N,
                                                           int max_samples, const int *chosen, int chain_offset, int n_local, const int *ids,
                                                           int qlo, int qhi, int max_lag, double *stats, double *halves, int *n_out)
{
  __shared__ double sbuf[32 * (SER_DIAG_SA + SER_DIAG_SB)]; /* moment partials [5][32 warps][32 lanes], then the staged chunks */
  __shared__ double s_mean[32], s_m1[32], s_m2[32];
  __shared__ int s_on[32];  /* quantity requested, and not constant in this chain */
  __shared__ int s_act[32]; /* its warp is still summing lags: only these traces are staged */
  __shared__ int s_eq1[32], s_eq2[32]; /* every sample of the first / last half equals that half's first one */
  const int c = blockIdx.x;
  const int local = local_chain(chosen[c], chain_offset, n_local, ids);
  if (local < 0) return;
  const int T = stored_samples(scal, local, max_samples);
  if (blockIdx.y == 0 && threadIdx.x == 0) n_out[c] = T;
  if (T < 4) return; /* the host refuses the call */
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, Q = 3 + N, n = T / 2;
  const int q0 = (qlo / 32 + blockIdx.y) * 32;
  const size_t row0 = (size_t)local * max_samples;
  const uint16_t *pi = samp_pi ? samp_pi + row0 * N : nullptr;
  const double *cdl = samp_cdl ? samp_cdl + row0 * 3 : nullptr;
  const double NaN = __longlong_as_double(0x7ff8000000000000LL);
  const int q = q0 + lane;
  const bool valid = q >= qlo && q < qhi;
  double *out = stats + ((size_t)c * Q + q) * 4, *hv = halves + ((size_t)c * Q + q) * 4;
  if (w == 0) { s_eq1[lane] = 1; s_eq2[lane] = 1; }
  __syncthreads();

  /* pass 1: sums over the trace and its halves (the middle sample of an odd T is in neither), min and max, and whether each half
   * is constant -- then its mean is its value and its variance 0 exactly, not the rounding residue of S / n */
  double s = 0.0, s1 = 0.0, s2 = 0.0, lo = INFINITY, hi = -INFINITY;
  const double f1 = valid ? diag_value(pi, cdl, N, q, 0) : 0.0, f2 = valid ? diag_value(pi, cdl, N, q, T - n) : 0.0;
  bool eq1 = true, eq2 = true;
  if (valid)
    for (int t = w; t < T; t += 32) {
      const double x = diag_value(pi, cdl, N, q, t);
      s += x;
      if (t < n) { s1 += x; eq1 = eq1 && x == f1; }
      if (t >= T - n) { s2 += x; eq2 = eq2 && x == f2; }
      lo = fmin(lo, x); hi = fmax(hi, x);
    }
  if (!eq1) atomicAnd(&s_eq1[lane], 0); /* an AND: the same result in any order */
  if (!eq2) atomicAnd(&s_eq2[lane], 0);
  double *ps = sbuf + threadIdx.x; /* partial [r][w][lane] at ps[r * 1024] */
  ps[0] = s; ps[1024] = s1; ps[2048] = s2; ps[3072] = lo; ps[4096] = hi;
  __syncthreads();
  if (w == 0) {
    double S = 0.0, S1 = 0.0, S2 = 0.0, L0 = INFINITY, H0 = -INFINITY;
    for (int u = 0; u < 32; u++) {
      const double *p = sbuf + u * 32 + lane;
      S += p[0]; S1 += p[1024]; S2 += p[2048]; L0 = fmin(L0, p[3072]); H0 = fmax(H0, p[4096]);
    }
    const bool constant = L0 == H0; /* gamma_0 = 0: the mean is the value itself, exactly */
    s_mean[lane] = constant ? L0 : S / T;
    s_m1[lane] = s_eq1[lane] ? f1 : S1 / n;
    s_m2[lane] = s_eq2[lane] ? f2 : S2 / n;
    s_on[lane] = valid && !constant;
  }
  __syncthreads();
  /* pass 2: centred squares about each part's own mean (zero for a constant quantity or half) */
  const double m = s_mean[lane], m1 = s_m1[lane], m2 = s_m2[lane];
  const bool var1 = !s_eq1[lane], var2 = !s_eq2[lane];
  double v = 0.0, v1 = 0.0, v2 = 0.0;
  if (s_on[lane])
    for (int t = w; t < T; t += 32) {
      const double x = diag_value(pi, cdl, N, q, t);
      v += (x - m) * (x - m);
      if (t < n && var1) v1 += (x - m1) * (x - m1);
      if (t >= T - n && var2) v2 += (x - m2) * (x - m2);
    }
  ps[0] = v; ps[1024] = v1; ps[2048] = v2;
  __syncthreads();
  if (w == 0 && valid) {
    double V = 0.0, V1 = 0.0, V2 = 0.0;
    for (int u = 0; u < 32; u++) {
      const double *p = sbuf + u * 32 + lane;
      V += p[0]; V1 += p[1024]; V2 += p[2048];
    }
    out[0] = m; out[1] = V / (T - 1);
    hv[0] = m1; hv[1] = V1 / (n - 1); hv[2] = m2; hv[3] = V2 / (n - 1);
  }

  /* autocovariances: warp w owns quantity q0 + w; lane l sums (x_t - m)(x_{t+k} - m) for k = k0 + l over t < T - k0 in t order */
  const int L = (max_lag > 0 && max_lag < T) ? max_lag : T;
  const int qw = q0 + w;
  bool on = s_on[w] != 0;
  double g0 = 0.0, psum = 0.0, pprev = INFINITY;
  int lags = 0;
  double *sA = sbuf, *sB = sbuf + 32 * SER_DIAG_SA;
  for (int k0 = 0;; k0 += 32) {
    if (lane == 0) s_act[w] = on;
    if (!__syncthreads_or(on)) break;
    double acc = 0.0;
    const int span = T - k0;
    for (int t0 = 0; t0 < span; t0 += SER_DIAG_TC) {
      __syncthreads();
      stage_lag_chunk(sA, sB, s_act, t0, k0, T, [&](int j, int t) { return diag_value(pi, cdl, N, q0 + j, t) - s_mean[j]; });
      __syncthreads();
      if (on) acc = lag_chunk_dot(sA, sB, w, lane, min(SER_DIAG_TC, span - t0), acc);
    }
    if (on) { /* Geyer's initial monotone sequence over this block's 16 pairs; every lane follows it, so `on` stays warp-uniform */
      if (k0 == 0) g0 = __shfl_sync(0xffffffffu, acc, 0) / T;
      for (int i = 0; i < 16; i++) {
        const double r0 = __shfl_sync(0xffffffffu, acc, 2 * i) / T / g0, r1 = __shfl_sync(0xffffffffu, acc, 2 * i + 1) / T / g0;
        if (k0 + 2 * i + 1 >= L) { on = false; break; } /* the pair needs both lags below L */
        double P = r0 + r1;
        if (!(P > 0.0)) { on = false; break; }
        P = fmin(P, pprev);
        pprev = P; psum += P; lags += 2;
      }
      if (k0 + 33 >= L || !(g0 >= DBL_MIN)) on = false;
    }
  }
  if (lane == 0 && qw >= qlo && qw < qhi) {
    double *o = stats + ((size_t)c * Q + qw) * 4;
    /* gamma_0 below DBL_MIN (a spread under ~1e-154, e.g. exp(c) at c ~ -745): the centred products underflow and rho_k means
     * nothing, so the ESS is undefined as for a constant quantity, not the floor that rho = NaN would give */
    const bool defined = s_on[w] != 0 && g0 >= DBL_MIN;
    o[2] = defined ? T / fmax(-1.0 + 2.0 * psum, 1.0 / log10((double)T)) : NaN;
    o[3] = defined ? (double)lags : 0.0;
  }
}

/* ------------------------------------------------------------------ posterior marginals (ser_run_marginals, DESIGN.md 3.8)
 * Histogram of item r over T samples: h[r][v] = #{t : x[t * stride + r] = v}, v in [0, bins).  pi: items = sites, stride N, N bins;
 * a, b: items = taxa (file order, as stored), stride M, N + 1 bins.  One thread owns one item's row, so no atomics are needed; the
 * loads of a sample row are coalesced (consecutive items are consecutive uint16_t).  The block's rows [r0, r0 + blockDim.x) are
 * contiguous in a [items][bins] slab: they are zeroed and written out as one coalesced span.  With s_rows (blockDim.x * bins ints
 * of dynamic shared memory) the counts are kept there; without, in the slab itself. */
__device__ void hist_tile(const uint16_t *x, int stride, int items, int bins, int T, int r0, int *slab, int *s_rows, bool add)
{
  const int nt = blockDim.x, n = min(nt, items - r0);
  const size_t cells = (size_t)n * bins;
  int *dst = slab + (size_t)r0 * bins, *h = s_rows ? s_rows : dst;
  if (s_rows || !add) {
    for (size_t e = threadIdx.x; e < cells; e += nt) h[e] = 0;
    __syncthreads();
  }
  if ((int)threadIdx.x < n) {
    int *row = h + (size_t)threadIdx.x * bins;
    const uint16_t *col = x + r0 + threadIdx.x;
    for (int t = 0; t < T; t++) row[col[(size_t)t * stride]]++;
  }
  if (s_rows) {
    __syncthreads();
    for (size_t e = threadIdx.x; e < cells; e += nt) dst[e] = add ? dst[e] + h[e] : h[e];
  }
}

/* pos [N][N]: the position histogram of every site over the chain's rows */
__global__ void ser_pos_hist_kernel(const uint16_t *samp_pi, const ChainScalars *scal, int N, int max_samples, SumSel sel, int use_smem,
                                    int *pos, size_t stride, int add)
{
  extern __shared__ int s_hist[];
  int T;
  const int local = sel_chain(sel, scal, blockIdx.x, blockIdx.y == 0 && threadIdx.x == 0, &T);
  if (local < 0) return;
  hist_tile(samp_pi + (size_t)local * max_samples * N, N, N, N, T, blockIdx.y * blockDim.x, pos + blockIdx.x * stride,
            use_smem ? s_hist : nullptr, add);
}

/* a_hist / b_hist [M][N+1] (blockIdx.z = 0 / 1; either may be nullptr): the histograms of every taxon's a and b over the chain's rows */
__global__ void ser_range_hist_kernel(const uint16_t *samp_a, const uint16_t *samp_b, const ChainScalars *scal, int N, int M, int max_samples,
                                      SumSel sel, int use_smem, int *a_hist, int *b_hist, size_t stride, int add)
{
  extern __shared__ int s_hist[];
  int *out = blockIdx.z ? b_hist : a_hist;
  if (!out) return;
  int T;
  const int local = sel_chain(sel, scal, blockIdx.x, blockIdx.y == 0 && threadIdx.x == 0, &T);
  if (local < 0) return;
  const uint16_t *x = (blockIdx.z ? samp_b : samp_a) + (size_t)local * max_samples * M;
  hist_tile(x, M, M, N + 1, T, blockIdx.y * blockDim.x, out + blockIdx.x * stride, use_smem ? s_hist : nullptr, add);
}

/* ------------------------------------------------------------------ diversity curves (ser_run_diversity, DESIGN.md 3.12)
 * Two stages over a pass of `rows` sample rows [t0, t0 + rows) of every chain (SER_DIV_CHUNK at most, so the scratch stays bounded):
 * stage 1 turns each sample row into its curves, u16 rows of scratch [k][rows][4][N] (D richness, O originations, E extinctions, then
 * D at the position of each site); stage 2 histograms every position's or site's column of them with hist_tile, bins = M + 1. */
#define SER_DIV_CHUNK 1024
#define SER_DIV_THREADS 256

/* Stage 1, one block per (row t0 + blockIdx.x, chain blockIdx.y).  The non-empty ranges' starts (at a) and stops (at b) are counted in
 * shared memory with integer atomics (the same in any order); D(p) = sum_{q <= p} (starts[q] - stops[q]) is a block scan taken
 * SER_DIV_THREADS positions at a time, O(p) = starts[p], E(p) = stops[p + 1]; the site row gathers D(pi_t(i)). */
__global__ void __launch_bounds__(SER_DIV_THREADS) ser_div_curve_kernel(const uint16_t *samp_a, const uint16_t *samp_b, const uint16_t *samp_pi,
                                                                        const ChainScalars *scal, int N, int M, int max_samples, SumSel sel,
                                                                        int t0, uint16_t *scratch)
{
  __shared__ int s_st[SER_MAX_SITES + 1], s_en[SER_MAX_SITES + 1], s_warp[SER_DIV_THREADS / 32];
  int T;
  const int local = sel_chain(sel, scal, blockIdx.y, false, &T), t = t0 + blockIdx.x;
  if (local < 0 || t >= T) return;
  for (int p = threadIdx.x; p <= N; p += blockDim.x) { s_st[p] = 0; s_en[p] = 0; }
  __syncthreads();
  const size_t row = (size_t)local * max_samples + t;
  const uint16_t *A = samp_a + row * M, *B = samp_b + row * M;
  for (int m = threadIdx.x; m < M; m += blockDim.x) {
    const int a = A[m], b = B[m];
    if (a < b) { atomicAdd(&s_st[a], 1); atomicAdd(&s_en[b], 1); }
  }
  __syncthreads();
  uint16_t *out = scratch + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 4 * N;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int carry = 0;
  for (int p0 = 0; p0 < N; p0 += blockDim.x) {
    const int p = p0 + threadIdx.x;
    const int o = p < N ? s_st[p] : 0, e = p < N ? s_en[p + 1] : 0;
    int v = p < N ? o - s_en[p] : 0;
    for (int d = 1; d < 32; d <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, v, d);
      if (lane >= d) v += y;
    }
    if (lane == 31) s_warp[warp] = v;
    __syncthreads();
    int before = carry;
    for (int w = 0; w < nw; w++) {
      const int s = s_warp[w];
      carry += s;
      if (w < warp) before += s;
    }
    if (p < N) { /* only this thread reads s_st[p]: it becomes D(p) */
      const int D = before + v;
      s_st[p] = D;
      out[p] = (uint16_t)D;
      out[N + p] = (uint16_t)o;
      out[2 * N + p] = (uint16_t)e;
    }
    __syncthreads();
  }
  const uint16_t *P = samp_pi + row * N;
  for (int i = threadIdx.x; i < N; i += blockDim.x) out[3 * N + i] = (uint16_t)s_st[P[i]];
}

/* Stage 2: output blockIdx.z (richness, originations, extinctions, site richness; nullptr: not wanted) of chain blockIdx.x, its rows
 * [blockIdx.y * blockDim.x, +blockDim.x) of [N][M + 1], over the pass's rows of that chain; add = 0 stores the slab, add = 1 adds. */
__global__ void ser_div_hist_kernel(const uint16_t *scratch, const ChainScalars *scal, int N, int M, SumSel sel, int t0, int rows, int use_smem,
                                    int *rich, int *orig, int *ext, int *site, size_t stride, int add)
{
  extern __shared__ int s_hist[];
  int *out = blockIdx.z == 0 ? rich : blockIdx.z == 1 ? orig : blockIdx.z == 2 ? ext : site;
  if (!out) return;
  int T;
  const int local = sel_chain(sel, scal, blockIdx.x, blockIdx.y == 0 && threadIdx.x == 0, &T);
  if (local < 0) return;
  const int n = min(max(T - t0, 0), rows);
  hist_tile(scratch + (size_t)blockIdx.x * rows * 4 * N + (size_t)blockIdx.z * N, 4 * N, N, M + 1, n, blockIdx.y * blockDim.x,
            out + blockIdx.x * stride, use_smem ? s_hist : nullptr, add);
}

/* ------------------------------------------------------------------ rank-normalised diagnostics (ser_run_rank_diagnostics, DESIGN.md 3.9)
 * The draws pool the chosen chains, ascending global id: sequence j is the first (j even) or the last (j odd) n = T/2 stored samples
 * of chosen chain j/2, draw (j, t) its row t or T - n + t (the middle row of an odd T is in neither), S = m n draws over m = 2k
 * sequences.  Series s of quantity q: 0 = z (the rank-normalised draws), 1 = z of the folded draws |x - median|, 2 = x,
 * 3 / 4 = 1{x <= q05} / 1{x <= q95}.  Sites get z from per-site tables built from the pooled position histogram; the three scalars
 * from two device sorts each.  No sum depends on the grid. */
struct RankSeq {
  const int *loc; /* local chain of each chosen chain, ascending global id */
  int T, n, m, max_samples;
};

__device__ __forceinline__ size_t rank_row(const RankSeq &r, int j, int t)
{
  return (size_t)r.loc[j >> 1] * r.max_samples + ((j & 1) ? r.T - r.n + t : t);
}

/* numpy's _lerp (numpy.quantile, method 'linear'), with no contraction */
__device__ __forceinline__ double np_lerp(double a, double b, double t)
{
  const double d = __dsub_rn(b, a);
  return t < 0.5 ? __dadd_rn(a, __dmul_rn(d, t)) : __dsub_rn(b, __dmul_rn(d, __dsub_rn(1.0, t)));
}

/* q05, q95 (numpy.quantile) and the median (numpy.median, S even) of S draws whose 0-based order statistic i is xs(i) */
template <class X>
__device__ void rank_quantiles(X xs, int S, double out[3])
{
  const double p[2] = {0.05, 0.95};
  for (int u = 0; u < 2; u++) {
    const double h = __dmul_rn((double)(S - 1), p[u]), j = floor(h);
    out[u] = np_lerp(xs((int)j), xs(min((int)j + 1, S - 1)), __dsub_rn(h, j));
  }
  out[2] = __dmul_rn(__dadd_rn(xs(S / 2 - 1), xs(S / 2)), 0.5);
}

/* z = Phi^-1((r - 3/8) / (S + 1/4)) of a value whose `ties` equal draws sit at the 0-based sorted positions [below, below + ties) */
__device__ __forceinline__ double rank_z(long long below, long long ties, int S)
{
  const double r = (double)below + (double)(ties + 1) * 0.5;
  return normcdfinv((r - 0.375) / ((double)S + 0.25));
}

/* the pooled position histogram hist [N][N] of the split rows: hist_tile over the m sequences in order (the first stores, the others add) */
__global__ void ser_rank_hist_kernel(const uint16_t *samp_pi, int N, RankSeq r, int use_smem, int *hist)
{
  extern __shared__ int s_hist[];
  for (int j = 0; j < r.m; j++)
    hist_tile(samp_pi + rank_row(r, j, 0) * N, N, N, N, r.n, blockIdx.x * blockDim.x, hist, use_smem ? s_hist : nullptr, j > 0);
}

/* dst[p] = sum_{v < p} get(v) for p <= len (dst[len] = the total), in integers; every thread of the block calls it */
template <class Get>
__device__ void block_scan_counts(Get get, int len, int *dst, int *part)
{
  const int per = (len + blockDim.x - 1) / blockDim.x, lo = min(len, (int)threadIdx.x * per), hi = min(len, lo + per);
  int s = 0;
  for (int p = lo; p < hi; p++) s += get(p);
  part[threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    int a = 0;
    for (int u = 0; u < (int)blockDim.x; u++) { const int v = part[u]; part[u] = a; a += v; }
    dst[len] = a;
  }
  __syncthreads();
  s = part[threadIdx.x];
  for (int p = lo; p < hi; p++) { dst[p] = s; s += get(p); }
  __syncthreads();
}

/* Site i = blockIdx.x from its row of the pooled histogram: z[i][p] and z_fold[i][p] of every position p held by a draw (0 elsewhere),
 * qs[3 + i] = q05, q95, median and out[3 + i][6..7] = q05, q95.  The folded value |p - med| is shared by p = med -/+ s (med an
 * integer) or floor(med) - s and floor(med) + 1 + s (med a half-integer): fold index s counts both, and the ranks of the folded draws
 * follow from the running counts over s. */
__global__ void __launch_bounds__(256) ser_rank_table_kernel(const int *hist, int N, int S, double *zt, double *zft, double *qs, double *out)
{
  __shared__ int s_h[SER_MAX_SITES], s_c[SER_MAX_SITES + 1], s_f[SER_MAX_SITES + 1], s_part[256];
  __shared__ double s_q[3];
  const int i = blockIdx.x;
  for (int p = threadIdx.x; p < N; p += blockDim.x) s_h[p] = hist[(size_t)i * N + p];
  __syncthreads();
  block_scan_counts([&](int p) { return s_h[p]; }, N, s_c, s_part);
  if (threadIdx.x == 0) {
    double v[3];
    rank_quantiles([&](int j) { /* the position holding order statistic j: the smallest p with s_c[p + 1] > j */
      int lo = 0, hi = N - 1;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (s_c[mid + 1] > j) hi = mid; else lo = mid + 1; }
      return (double)lo;
    }, S, v);
    for (int u = 0; u < 3; u++) { s_q[u] = v[u]; qs[(size_t)(3 + i) * 3 + u] = v[u]; }
    out[(size_t)(3 + i) * 8 + 6] = v[0]; out[(size_t)(3 + i) * 8 + 7] = v[1];
  }
  __syncthreads();
  const double med = s_q[2];
  const int m0 = (int)floor(med), half = med != (double)m0;
  auto fold_count = [&](int s) {
    const int lo = m0 - s, hi = half ? m0 + 1 + s : m0 + s;
    return (lo >= 0 ? s_h[lo] : 0) + (hi != lo && hi < N ? s_h[hi] : 0);
  };
  block_scan_counts(fold_count, N, s_f, s_part);
  for (int p = threadIdx.x; p < N; p += blockDim.x) {
    const int h = s_h[p], s = p <= m0 ? m0 - p : p - m0 - half;
    zt[(size_t)i * N + p] = h ? rank_z(s_c[p], h, S) : 0.0;
    zft[(size_t)i * N + p] = h ? rank_z(s_f[s], fold_count(s), S) : 0.0;
  }
}

/* keys[q][s] = x of draw s = j n + t of scalar q = blockIdx.y (fold: |x - median_q|), vals[q][s] = s */
__global__ void ser_rank_gather_kernel(const double *samp_cdl, RankSeq r, const double *qs, int fold, double *keys, int *vals)
{
  const int q = blockIdx.y, S = r.m * r.n;
  for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < S; s += gridDim.x * blockDim.x) {
    const int j = s / r.n, t = s - j * r.n;
    const double x = diag_value(nullptr, samp_cdl + rank_row(r, j, t) * 3, 0, q, 0);
    keys[(size_t)q * S + s] = fold ? fabs(__dsub_rn(x, qs[q * 3 + 2])) : x;
    vals[(size_t)q * S + s] = s;
  }
}

/* From the sorted keys of scalar q = blockIdx.y: z[q][draw] of every draw from its average rank (ties = equal doubles, found by binary
 * search), and unless fold, qs[q] = q05, q95, median and out[q][6..7] = q05, q95 */
__global__ void ser_rank_scalar_kernel(const double *keys, const int *vals, int S, int fold, double *z, double *qs, double *out)
{
  const int q = blockIdx.y;
  const double *k = keys + (size_t)q * S;
  for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < S; s += gridDim.x * blockDim.x) {
    const double x = k[s];
    int lo = 0, hi = s; /* first index whose key equals x */
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (k[mid] < x) lo = mid + 1; else hi = mid; }
    const int a = lo;
    lo = s + 1; hi = S; /* one past the last */
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (k[mid] > x) hi = mid; else lo = mid + 1; }
    z[(size_t)q * S + vals[(size_t)q * S + s]] = rank_z(a, lo - a, S);
  }
  if (!fold && blockIdx.x == 0 && threadIdx.x == 0) {
    double v[3];
    rank_quantiles([&](int j) { return k[j]; }, S, v);
    for (int u = 0; u < 3; u++) qs[q * 3 + u] = v[u];
    out[q * 8 + 6] = v[0]; out[q * 8 + 7] = v[1];
  }
}

/* What the series of a quantity read: the store, the site tables z / z_fold [N][N], the scalar traces z / z_fold [3][S] (draw order) and
 * qs [3 + N][3] = q05, q95, median */
struct RankSrc {
  const uint16_t *pi;
  const double *cdl, *zt, *zft, *zs, *zfs, *qs;
  int N;
};

__device__ __forceinline__ double rank_value(const RankSrc &s, const RankSeq &r, int series, int q, int j, int t)
{
  const size_t row = rank_row(r, j, t);
  if (series < 2) {
    if (q < 3) return (series ? s.zfs : s.zs)[(size_t)q * r.m * r.n + (size_t)j * r.n + t];
    return (series ? s.zft : s.zt)[(size_t)(q - 3) * s.N + s.pi[row * s.N + q - 3]];
  }
  const double x = q < 3 ? diag_value(nullptr, s.cdl + row * 3, s.N, q, 0) : (double)s.pi[row * s.N + q - 3];
  return series == 2 ? x : (x <= s.qs[q * 3 + series - 3] ? 1.0 : 0.0);
}

/* R-hat and ESS of series blockIdx.y over the m sequences, one block of 32 warps per 32 consecutive quantities.  Pass 1: lane = quantity,
 * warp w takes sequences w, w + 32, ..., each summed in t order: its mean (its value when constant) and variance (divisor n - 1; 0 when
 * constant) go to seq [5][3+N][m][2].  Warp 0 then pools them in sequence order: W, B/n, R-hat (series 0, 1 into out[q][0..1]) and
 * var+.  Pass 2 (not for series 1): warp w owns quantity q0 + w, lane l sums lag k0 + l over sequence j = 0 .. m-1, then t, about each
 * sequence's own mean, staged as in ser_diag_kernel; after each 32-lag block the warp walks Stan's loop on rho(k0 .. k0 + 31) and stops
 * where the loop stops.  ESS goes to out[q][2..5] (series 0, 2, 3, 4). */
__global__ void __launch_bounds__(1024, 1) ser_rank_ess_kernel(RankSrc src, RankSeq r, int qlo, int qhi, double *seq, double *out)
{
  __shared__ double sbuf[32 * (SER_DIAG_SA + SER_DIAG_SB)];
  __shared__ double s_W[32], s_varp[32], s_cm[32];
  __shared__ int s_on[32], s_act[32];
  const int series = blockIdx.y, lane = threadIdx.x & 31, w = threadIdx.x >> 5, Q = 3 + src.N, m = r.m, n = r.n;
  const int q0 = (qlo / 32 + blockIdx.x) * 32, q = q0 + lane, field = series == 0 ? 2 : series + 1;
  const bool valid = q >= qlo && q < qhi;
  const double NaN = __longlong_as_double(0x7ff8000000000000LL);
  if (valid)
    for (int j = w; j < m; j += 32) {
      double s = 0.0, lo = INFINITY, hi = -INFINITY;
      for (int t = 0; t < n; t++) {
        const double x = rank_value(src, r, series, q, j, t);
        s += x; lo = fmin(lo, x); hi = fmax(hi, x);
      }
      const double mu = lo == hi ? lo : s / n;
      double v = 0.0;
      if (lo != hi)
        for (int t = 0; t < n; t++) { const double d = rank_value(src, r, series, q, j, t) - mu; v += d * d; }
      double *o = seq + (((size_t)series * Q + q) * m + j) * 2;
      o[0] = mu; o[1] = v / (n - 1);
    }
  __syncthreads();
  if (w == 0) {
    double W = 0.0, M = 0.0, Bn = 0.0, mlo = INFINITY, mhi = -INFINITY;
    const double *o = seq + ((size_t)series * Q + q) * m * 2;
    if (valid) {
      for (int j = 0; j < m; j++) { W += o[2 * j + 1]; M += o[2 * j]; mlo = fmin(mlo, o[2 * j]); mhi = fmax(mhi, o[2 * j]); }
      W /= m;
      if (mlo != mhi) { /* equal sequence means: B = 0 exactly, not the residue of their mean */
        const double mbar = M / m;
        for (int j = 0; j < m; j++) { const double d = o[2 * j] - mbar; Bn += d * d; }
        Bn /= m - 1;
      }
    }
    const double varp = W * (n - 1.0) / n + Bn;
    if (valid && series < 2) out[(size_t)q * 8 + series] = W > 0.0 ? sqrt(((n - 1.0) / n * W + Bn) / W) : Bn > 0.0 ? INFINITY : NaN;
    if (valid && series != 1 && !(varp > 0.0)) out[(size_t)q * 8 + field] = NaN; /* every draw equal */
    s_W[lane] = W; s_varp[lane] = varp;
    s_on[lane] = valid && series != 1 && varp > 0.0;
  }
  __syncthreads();

  /* Stan's loop, kept warp-uniform: (pe, po) is the last pair read (rho(t-1), rho(t)), stored when pe + po >= 0; reading the next pair
   * commits it, monotonised against the previous committed pair, into psum */
  const int qw = q0 + w;
  bool on = s_on[w] != 0;
  const double Wq = s_W[w], varp = s_varp[w], mn = (double)m * n;
  double pe = 1.0, po = 0.0, psum = 0.0, pprev = 0.0;
  bool stored = true, first = true;
  int t = 1;
  double *sA = sbuf, *sB = sbuf + 32 * SER_DIAG_SA;
  for (int k0 = 0;; k0 += 32) {
    if (lane == 0) s_act[w] = on;
    if (!__syncthreads_or(on)) break;
    double acc = 0.0;
    const int span = n - k0;
    for (int j = 0; j < m; j++) {
      if (threadIdx.x < 32) /* read by the staging after the barrier below; the previous staging is behind the last barrier */
        s_cm[threadIdx.x] = s_act[threadIdx.x] ? seq[(((size_t)series * Q + q0 + threadIdx.x) * m + j) * 2] : 0.0;
      for (int t0 = 0; t0 < span; t0 += SER_DIAG_TC) {
        __syncthreads();
        stage_lag_chunk(sA, sB, s_act, t0, k0, n, [&](int jq, int tt) { return rank_value(src, r, series, q0 + jq, j, tt) - s_cm[jq]; });
        __syncthreads();
        if (on) acc = lag_chunk_dot(sA, sB, w, lane, min(SER_DIAG_TC, span - t0), acc);
      }
    }
    if (on) {
      const double rho = 1.0 - (Wq - acc / mn) / varp; /* rho(k0 + lane) */
      if (k0 == 0) po = __shfl_sync(0xffffffffu, rho, 1);
      for (;;) {
        if (!(t < n - 3 && pe + po > 0.0)) { on = false; break; }
        if (t + 1 >= k0 + 32) break; /* the next pair is in the next lag block */
        const double e = __shfl_sync(0xffffffffu, rho, t + 1 - k0), o = __shfl_sync(0xffffffffu, rho, t + 2 - k0);
        double P = pe + po;
        if (!first && P > pprev) P = pprev;
        first = false; psum += P; pprev = P;
        pe = e; po = o; stored = e + o >= 0.0;
        t += 2;
      }
    }
  }
  if (lane == 0 && s_on[w]) {
    const double last = (pe > 0.0 || stored) ? pe : 0.0; /* rho[max_t + 1] */
    const double tau = fmax(-1.0 + 2.0 * psum + last, 1.0 / log10(mn));
    out[(size_t)qw * 8 + field] = mn / tau;
  }
}

/* ------------------------------------------------------------------ streaming accumulators (ser_run_accumulate)
 * On an accumulating run the sample store is a window of max_samples rows per chain.  After every sweep launch of w sampling calls
 * the summary kernels above add the window's rows of EVERY local chain into that chain's accumulator record; the getters turn the
 * records into what the one-shot kernels compute from a store that holds all samples, with the kernels below. */

#define SER_ACC_ALL \
  (SER_ACC_PO | SER_ACC_SUMS | SER_ACC_AB | SER_ACC_ALIVE | SER_ACC_POS | SER_ACC_RANGE | SER_ACC_TAXA | SER_ACC_CD | SER_ACC_DIV)

/* One local chain's accumulator record: int32 offsets of the parts the flags `what` select, in this order, and the record's length.
 * The run holds [n_local][ints]; a checkpoint record holds the same ints in the same order.
 *   po [N][N] (SER_ACC_PO; diagonal 0), pi [N] (SER_ACC_SUMS or SER_ACC_AB), asum [M], bsum [M] (SER_ACC_AB),
 *   alive [N][M] (SER_ACC_ALIVE; the difference slab), pos [N][N] (SER_ACC_POS), range [2][M][N+1] (SER_ACC_RANGE; a, then b),
 *   taxa [4][M][M] (SER_ACC_TAXA; first, last, precedes, coexist),
 *   cd: f64 c_sum, d_sum [R] as pairs of int32 words, then c_hist, d_hist [R][SER_CD_BINS] (SER_ACC_CD; R = M on a manycd run, else 1),
 *   div [4][N][M+1] (SER_ACC_DIV; richness, originations, extinctions, site richness: an even length, so the alignment below holds).
 * Under SER_ACC_CD alone the part's start and the record's length are rounded up to an even number of words, so every double is
 * 8-byte aligned in the run's records; records without the flag keep their length, and checkpoint files their bytes. */
struct AccLayout {
  size_t po, pi, asum, bsum, alive, pos, range, taxa, cd, div, ints;
};
__host__ __device__ inline AccLayout acc_layout(int N, int M, int manycd, int what)
{
  AccLayout L;
  const size_t n = N, m = M, cdr = manycd ? M : 1;
  size_t o = 0;
  L.po = o; o += (what & SER_ACC_PO) ? n * n : 0;
  L.pi = o; o += (what & (SER_ACC_SUMS | SER_ACC_AB)) ? n : 0;
  L.asum = o; o += (what & SER_ACC_AB) ? m : 0;
  L.bsum = o; o += (what & SER_ACC_AB) ? m : 0;
  L.alive = o; o += (what & SER_ACC_ALIVE) ? n * m : 0;
  L.pos = o; o += (what & SER_ACC_POS) ? n * n : 0;
  L.range = o; o += (what & SER_ACC_RANGE) ? 2 * m * (n + 1) : 0;
  L.taxa = o; o += (what & SER_ACC_TAXA) ? 4 * m * m : 0;
  if (what & SER_ACC_CD) o += o & 1;
  L.cd = o; o += (what & SER_ACC_CD) ? 4 * cdr + 2 * cdr * SER_CD_BINS : 0;
  L.div = o; o += (what & SER_ACC_DIV) ? 4 * n * (m + 1) : 0;
  L.ints = o;
  return L;
}

/* The getters of an accumulating run read the records of the chosen chains the run holds (sel: rows = INT_MAX, so T = all samples
 * taken since accumulation began); `acc` points at the part in local chain 0's record, records are `per_chain` ints apart. */

/* counts [k][N][N]: the pair-order part with the diagonal -T */
__global__ void ser_po_acc_out_kernel(const int *acc, size_t per_chain, const ChainScalars *scal, int N, SumSel sel, int *counts)
{
  int T;
  const int local = sel_chain(sel, scal, blockIdx.y, blockIdx.x == 0 && threadIdx.x == 0, &T);
  if (local < 0) return;
  const size_t nn = (size_t)N * N;
  for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < nn; q += (size_t)gridDim.x * blockDim.x)
    counts[blockIdx.y * nn + q] = (q / N == q % N) ? -T : acc[local * per_chain + q];
}

/* the pi, a and b sums (a_sum / b_sum may be nullptr) and corr_num[c] = sum_i i * pi_sum[c][i] */
__global__ void ser_posterior_acc_out_kernel(const int *pi_acc, const int *a_acc, const int *b_acc, size_t per_chain, const ChainScalars *scal,
                                             int N, int M, SumSel sel, long long *corr_num, int *pi_sum, int *a_sum, int *b_sum)
{
  __shared__ unsigned long long s_corr;
  int T;
  const int local = sel_chain(sel, scal, blockIdx.x, threadIdx.x == 0, &T);
  if (local < 0) return;
  if (threadIdx.x == 0) s_corr = 0;
  __syncthreads();
  const size_t src = local * per_chain;
  long long s = 0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const int v = pi_acc[src + i];
    pi_sum[(size_t)blockIdx.x * N + i] = v;
    s += (long long)i * v;
  }
  for (int m = threadIdx.x; m < M; m += blockDim.x) {
    if (a_sum) a_sum[(size_t)blockIdx.x * M + m] = a_acc[src + m];
    if (b_sum) b_sum[(size_t)blockIdx.x * M + m] = b_acc[src + m];
  }
  atomicAdd(&s_corr, (unsigned long long)s); /* an integer sum: the same in any order */
  __syncthreads();
  if (threadIdx.x == 0) corr_num[blockIdx.x] = (long long)s_corr;
}

/* alive [k][N][M]: the running sum of the difference slab down the positions */
__global__ void ser_alive_acc_out_kernel(const int *diff, size_t per_chain, const ChainScalars *scal, int N, int M, SumSel sel, int *alive)
{
  int T;
  const int local = sel_chain(sel, scal, blockIdx.x, blockIdx.y == 0 && threadIdx.x == 0, &T);
  if (local < 0) return;
  const int m = blockIdx.y * blockDim.x + threadIdx.x;
  if (m >= M) return;
  const int *src = diff + local * per_chain + m;
  int *col = alive + (size_t)blockIdx.x * N * M + m;
  int acc = 0;
  for (int j = 0; j < N; j++) { acc += src[(size_t)j * M]; col[(size_t)j * M] = acc; }
}

/* histogram part z (blockIdx.z) of `cells` ints into out_z [k][cells] (nullptr: not wanted), chosen chain blockIdx.y */
__global__ void ser_hist_acc_out_kernel(const int *acc, size_t per_chain, size_t cells, const ChainScalars *scal, SumSel sel, int *out0,
                                        int *out1)
{
  int *out = blockIdx.z ? out1 : out0;
  if (!out) return;
  int T;
  const int local = sel_chain(sel, scal, blockIdx.y, blockIdx.x == 0 && threadIdx.x == 0, &T);
  if (local < 0) return;
  const int *src = acc + local * per_chain + blockIdx.z * cells;
  for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < cells; q += (size_t)gridDim.x * blockDim.x)
    out[blockIdx.y * cells + q] = src[q];
}

/* ------------------------------------------------------------------ micro-benchmarks */
__global__ void mb_fp64_kernel(double *out, int iters)
{
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double m = 1.0000001, c = 1e-7;
  for (int i = 0; i < iters; i++) {
    a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
    a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}
__global__ void mb_lds_kernel(unsigned *out, int iters)
{
  __shared__ uint4 buf[1024];
  buf[threadIdx.x] = make_uint4(threadIdx.x, 1, 2, 3);
  __syncthreads();
  uint4 acc = make_uint4(0, 0, 0, 0);
  int idx = threadIdx.x;
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int u = 0; u < 8; u++) {
      const uint4 v = buf[(idx + u * 32) & 1023];
      acc.x += v.x; acc.y ^= v.y; acc.z += v.z; acc.w ^= v.w;
    }
    idx = (idx + acc.y) & 1023;
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = acc.x + acc.y + acc.z + acc.w;
}
__global__ void mb_popc_kernel(unsigned *out, int iters)
{
  unsigned x0 = threadIdx.x + 1, x1 = x0 * 3, x2 = x0 * 5, x3 = x0 * 7, s0 = 0, s1 = 0, s2 = 0, s3 = 0;
  for (int i = 0; i < iters; i++) {
    s0 += __popc(x0 ^ s3); s1 += __popc(x1 ^ s0); s2 += __popc(x2 ^ s1); s3 += __popc(x3 ^ s2);
    s0 += __popc(x0 + s2); s1 += __popc(x1 + s3); s2 += __popc(x2 + s0); s3 += __popc(x3 + s1);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = s0 + s1 + s2 + s3;
}
