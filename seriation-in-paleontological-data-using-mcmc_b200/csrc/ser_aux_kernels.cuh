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

/* pair-order counts (script.py:178-189) for one chosen chain per blockIdx.z, one 32 x 32 tile per block.  T = the CHOSEN
 * chain's own sample count.  Only the owner of a chosen chain writes its slab -- to every destination (peer stores: the
 * slabs are disjoint, so no reduction is needed). */
__global__ void __launch_bounds__(256) ser_po_kernel(const uint16_t *samp_pi, const ChainScalars *scal, int N, int max_samples,
                                                      const int *chosen, int chain_offset, int n_local, const int *ids, PeerPtrs dst)
{
  const int local = local_chain(chosen[blockIdx.z], chain_offset, n_local, ids);
  if (local < 0) return;
  const int T = stored_samples(scal, local, max_samples);
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
    const int v = (i == j) ? -T : c[r];
    for (int q = 0; q < dst.n; q++) ((int *)dst.p[q])[((size_t)blockIdx.z * N + i) * N + j] = v;
  }
}

/* posterior sums over the stored samples of one chosen chain per block (script.py:129-152, :230-276) */
__global__ void ser_posterior_kernel(const uint16_t *samp_pi, const uint16_t *samp_a, const uint16_t *samp_b, const ChainScalars *scal,
                                     int N, int M, int max_samples, const int *chosen, int chain_offset, int n_local, const int *ids,
                                     long long *corr_num, int *pi_sum, int *a_sum, int *b_sum, int *n_out)
{
  const int local = local_chain(chosen[blockIdx.x], chain_offset, n_local, ids);
  if (local < 0) return;
  const int n_samples = stored_samples(scal, local, max_samples);
  if (threadIdx.x == 0 && n_out) n_out[blockIdx.x] = n_samples;
  const size_t base = (size_t)local * max_samples;
  long long s = 0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    int acc = 0;
    for (int t = 0; t < n_samples; t++) acc += samp_pi[(base + t) * N + i];
    pi_sum[(size_t)blockIdx.x * N + i] = acc;
    s += (long long)i * acc;
  }
  if (a_sum && samp_a)
    for (int m = threadIdx.x; m < M; m += blockDim.x) {
      int sa = 0, sb = 0;
      for (int t = 0; t < n_samples; t++) { sa += samp_a[(base + t) * M + m]; sb += samp_b[(base + t) * M + m]; }
      a_sum[(size_t)blockIdx.x * M + m] = sa;
      if (b_sum) b_sum[(size_t)blockIdx.x * M + m] = sb;
    }
  atomicAdd((unsigned long long *)&corr_num[blockIdx.x], (unsigned long long)s);
}

/* alive[c][j][m] = #{t : a_t(m) <= j <= b_t(m)} over the stored samples of chosen chain c
 * (script.py:321-329; closed at b, as the reference tests it).  One thread per taxon: +1 / -1
 * marks at a and b+1 in its own column of the slab, then a running sum down the positions. */
__global__ void ser_alive_kernel(const uint16_t *samp_a, const uint16_t *samp_b, const ChainScalars *scal, int N, int M, int max_samples,
                                 const int *chosen, int chain_offset, int n_local, const int *ids, int *alive, int *n_out)
{
  const int local = local_chain(chosen[blockIdx.x], chain_offset, n_local, ids);
  if (local < 0) return;
  const int n_samples = stored_samples(scal, local, max_samples);
  if (blockIdx.y == 0 && threadIdx.x == 0 && n_out) n_out[blockIdx.x] = n_samples;
  const int m = blockIdx.y * blockDim.x + threadIdx.x;
  if (m >= M) return;
  const size_t base = (size_t)local * max_samples;
  int *col = alive + (size_t)blockIdx.x * N * M + m;
  for (int j = 0; j < N; j++) col[(size_t)j * M] = 0;
  for (int t = 0; t < n_samples; t++) {
    const int a = samp_a[(base + t) * M + m], b = samp_b[(base + t) * M + m];
    if (a < N) col[(size_t)a * M] += 1;
    if (b + 1 < N) col[(size_t)(b + 1) * M] -= 1;
  }
  int acc = 0;
  for (int j = 0; j < N; j++) { acc += col[(size_t)j * M]; col[(size_t)j * M] = acc; }
}

/* ------------------------------------------------------------------ streaming accumulators (ser_run_accumulate)
 * On an accumulating run the sample store is a window of max_samples rows per chain.  After every sweep launch of w
 * sampling calls these kernels add rows [0, w) of EVERY local chain's window into per-chain totals; the getters below
 * turn the totals into what the one-shot kernels above compute from a store that holds all samples. */

/* rows of the window a chain filled in the last launch (fewer than w only when its replay tape ran out) */
__device__ __forceinline__ int window_rows(const ChainScalars *scal, int local, int sample_base, int w)
{
  const int n = scal[local].n_samples - sample_base;
  return n < 0 ? 0 : n < w ? n : w;
}

/* pair-order tiles of every local chain (blockIdx.z) added into acc [n_local][N][N]; the diagonal stays 0 */
__global__ void __launch_bounds__(256) ser_po_accum_kernel(const uint16_t *samp_pi, const ChainScalars *scal, int N, int max_samples,
                                                            int sample_base, int w, int *acc)
{
  const int local = blockIdx.z;
  const int T = window_rows(scal, local, sample_base, w);
  if (T == 0) return;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int i0 = blockIdx.y * 32, j0 = blockIdx.x * 32;
  int c[4] = {0, 0, 0, 0};
  po_tile(samp_pi + (size_t)local * max_samples * N, N, T, i0, j0, c);
  const int j = j0 + tx;
  if (j >= N) return;
  int *slab = acc + (size_t)local * N * N;
#pragma unroll
  for (int r = 0; r < 4; r++) {
    const int i = i0 + ty + 8 * r;
    if (i < N) slab[(size_t)i * N + j] += c[r];
  }
}

/* sum_t pi_t into pi_acc [n_local][N], and sum_t a_t / b_t into a_acc / b_acc [n_local][M] when given; one chain per block */
__global__ void ser_posterior_accum_kernel(const uint16_t *samp_pi, const uint16_t *samp_a, const uint16_t *samp_b, const ChainScalars *scal,
                                           int N, int M, int max_samples, int sample_base, int w, int *pi_acc, int *a_acc, int *b_acc)
{
  const int local = blockIdx.x;
  const int T = window_rows(scal, local, sample_base, w);
  const size_t base = (size_t)local * max_samples;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    int acc = 0;
    for (int t = 0; t < T; t++) acc += samp_pi[(base + t) * N + i];
    pi_acc[(size_t)local * N + i] += acc;
  }
  if (a_acc)
    for (int m = threadIdx.x; m < M; m += blockDim.x) {
      int sa = 0, sb = 0;
      for (int t = 0; t < T; t++) { sa += samp_a[(base + t) * M + m]; sb += samp_b[(base + t) * M + m]; }
      a_acc[(size_t)local * M + m] += sa;
      b_acc[(size_t)local * M + m] += sb;
    }
}

/* +1 at a, -1 at b+1 of every window row into the difference slab diff [n_local][N][M]; one thread per taxon */
__global__ void ser_alive_accum_kernel(const uint16_t *samp_a, const uint16_t *samp_b, const ChainScalars *scal, int N, int M, int max_samples,
                                       int sample_base, int w, int *diff)
{
  const int local = blockIdx.x, m = blockIdx.y * blockDim.x + threadIdx.x;
  if (m >= M) return;
  const int T = window_rows(scal, local, sample_base, w);
  const size_t base = (size_t)local * max_samples;
  int *col = diff + (size_t)local * N * M + m;
  for (int t = 0; t < T; t++) {
    const int a = samp_a[(base + t) * M + m], b = samp_b[(base + t) * M + m];
    if (a < N) col[(size_t)a * M] += 1;
    if (b + 1 < N) col[(size_t)(b + 1) * M] -= 1;
  }
}

/* getters of an accumulating run: the slab of every chosen chain the run holds, T = all samples taken since accumulation began */
__global__ void ser_po_acc_out_kernel(const int *acc, const ChainScalars *scal, int N, const int *chosen, int chain_offset, int n_local,
                                      const int *ids, int *counts)
{
  const int local = local_chain(chosen[blockIdx.y], chain_offset, n_local, ids);
  if (local < 0) return;
  const int T = scal[local].n_samples;
  const size_t nn = (size_t)N * N;
  for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < nn; q += (size_t)gridDim.x * blockDim.x)
    counts[blockIdx.y * nn + q] = (q / N == q % N) ? -T : acc[local * nn + q];
}

__global__ void ser_posterior_acc_out_kernel(const int *pi_acc, const int *a_acc, const int *b_acc, const ChainScalars *scal, int N, int M,
                                             const int *chosen, int chain_offset, int n_local, const int *ids,
                                             long long *corr_num, int *pi_sum, int *a_sum, int *b_sum, int *n_out)
{
  const int local = local_chain(chosen[blockIdx.x], chain_offset, n_local, ids);
  if (local < 0) return;
  if (threadIdx.x == 0) n_out[blockIdx.x] = scal[local].n_samples;
  long long s = 0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const int v = pi_acc[(size_t)local * N + i];
    pi_sum[(size_t)blockIdx.x * N + i] = v;
    s += (long long)i * v;
  }
  if (a_sum)
    for (int m = threadIdx.x; m < M; m += blockDim.x) {
      a_sum[(size_t)blockIdx.x * M + m] = a_acc[(size_t)local * M + m];
      if (b_sum) b_sum[(size_t)blockIdx.x * M + m] = b_acc[(size_t)local * M + m];
    }
  atomicAdd((unsigned long long *)&corr_num[blockIdx.x], (unsigned long long)s);
}

/* running sum of the difference slab down the positions */
__global__ void ser_alive_acc_out_kernel(const int *diff, const ChainScalars *scal, int N, int M, const int *chosen, int chain_offset,
                                         int n_local, const int *ids, int *alive, int *n_out)
{
  const int local = local_chain(chosen[blockIdx.x], chain_offset, n_local, ids);
  if (local < 0) return;
  if (blockIdx.y == 0 && threadIdx.x == 0) n_out[blockIdx.x] = scal[local].n_samples;
  const int m = blockIdx.y * blockDim.x + threadIdx.x;
  if (m >= M) return;
  const int *src = diff + (size_t)local * N * M + m;
  int *col = alive + (size_t)blockIdx.x * N * M + m;
  int acc = 0;
  for (int j = 0; j < N; j++) { acc += src[(size_t)j * M]; col[(size_t)j * M] = acc; }
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
