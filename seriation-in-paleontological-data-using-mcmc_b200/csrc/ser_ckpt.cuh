/* ser_ckpt.cuh -- checkpoint files: every chain of a run written to a file and read back into another run, bit for bit.
 * Part of the single translation unit ser_kernels.cu (included last).  This is the only module that knows the format;
 * DESIGN.md section 3.6 describes it.
 *
 * A file is header | chain table | records, little-endian, every field of explicit width:
 *   header   SER_CKPT_HEADER bytes: magic "SERCKPT\0", u32 version, u32 header size, i32 N, M, nh, mode, u64 dataset
 *            fingerprint, u32 seed, i32 sweeps_per_call, manycd, store, max_samples, SER_ACC_* flags, i64 calls_done,
 *            i32 n_samples, sample_base, rows, n_chains, u64 record size, u64 checksum of the bytes before it
 *   table    i32 global chain id [n_chains], strictly ascending, zero-padded to 8 bytes, u64 checksum
 *   records  one per chain in table order, each record_size bytes and ending with the u64 checksum of the bytes before it
 * A record holds the live state as named fields (ckpt_layout below; a, b and per-taxon c, d in taxon order, whatever
 * column order the run keeps them in), then the stored sample rows and the accumulator slabs as the run holds them.
 * What a run derives from that state is rebuilt: the bit columns (SER_FLAG_COLUMNS is cleared, so the sweep kernel builds
 * them from rpi), and done[] / chunks_done restart from zero as after ser_run_init.  So the same chains in the same state
 * give the same bytes whatever the sharding or the sweep path. */
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <cerrno>
#include <string>

static_assert(__BYTE_ORDER__ == __ORDER_LITTLE_ENDIAN__, "records are written in the device's byte order, which is little-endian");

#define SER_CKPT_VERSION 1u
#define SER_CKPT_HEADER 104
#define SER_CKPT_SCALARS 168                 /* bytes of the named scalar fields at the start of a record */
#define SER_CKPT_STAGING (256ull << 20)      /* pinned host bytes a save or load stages through, whatever the run size */

/* FNV-1a over 64-bit little-endian words (every length hashed is a multiple of 8): a change in one word always changes
 * the result, because each step is a bijection of the running value */
static uint64_t ckpt_hash(const void *data, size_t bytes)
{
  const unsigned char *p = (const unsigned char *)data;
  uint64_t h = 0xcbf29ce484222325ull;
  for (size_t i = 0; i + 8 <= bytes; i += 8) {
    uint64_t w;
    memcpy(&w, p + i, 8);
    h = (h ^ w) * 0x100000001b3ull;
  }
  return h;
}

/* X as 0/1 cells, row-major, then the hard flags, zero-padded to whole words */
static uint64_t ckpt_dataset_fingerprint(const ser_dataset *ds)
{
  const size_t nm = (size_t)ds->N * ds->M, n = nm + ds->N;
  std::vector<unsigned char> cells((n + 7) / 8 * 8, 0);
  for (size_t i = 0; i < nm; i++) cells[i] = ds->X[i] != 0;
  for (int i = 0; i < ds->N; i++) cells[nm + i] = ds->hard[i] != 0;
  return ckpt_hash(cells.data(), cells.size());
}

struct CkptHeader {
  int32_t N, M, nh, mode;
  uint64_t fingerprint;
  uint32_t seed;
  int32_t sweeps_per_call, manycd, store, max_samples, acc;
  int64_t calls_done;
  int32_t n_samples, sample_base, rows, n_chains;
  uint64_t record_size;
};

static void put_le(unsigned char *b, uint64_t v, int bytes) { for (int i = 0; i < bytes; i++) b[i] = (unsigned char)(v >> (8 * i)); }
static uint64_t get_le(const unsigned char *b, int bytes)
{
  uint64_t v = 0;
  for (int i = 0; i < bytes; i++) v |= (uint64_t)b[i] << (8 * i);
  return v;
}

static void ckpt_encode_header(const CkptHeader &h, unsigned char b[SER_CKPT_HEADER])
{
  memset(b, 0, SER_CKPT_HEADER);
  memcpy(b, "SERCKPT", 8);
  put_le(b + 8, SER_CKPT_VERSION, 4); put_le(b + 12, SER_CKPT_HEADER, 4);
  put_le(b + 16, (uint32_t)h.N, 4); put_le(b + 20, (uint32_t)h.M, 4); put_le(b + 24, (uint32_t)h.nh, 4); put_le(b + 28, (uint32_t)h.mode, 4);
  put_le(b + 32, h.fingerprint, 8);
  put_le(b + 40, h.seed, 4); put_le(b + 44, (uint32_t)h.sweeps_per_call, 4); put_le(b + 48, (uint32_t)h.manycd, 4);
  put_le(b + 52, (uint32_t)h.store, 4); put_le(b + 56, (uint32_t)h.max_samples, 4); put_le(b + 60, (uint32_t)h.acc, 4);
  put_le(b + 64, (uint64_t)h.calls_done, 8);
  put_le(b + 72, (uint32_t)h.n_samples, 4); put_le(b + 76, (uint32_t)h.sample_base, 4); put_le(b + 80, (uint32_t)h.rows, 4);
  put_le(b + 84, (uint32_t)h.n_chains, 4);
  put_le(b + 88, h.record_size, 8);
  put_le(b + 96, ckpt_hash(b, 96), 8);
}

static void ckpt_decode_header(const unsigned char b[SER_CKPT_HEADER], CkptHeader *h)
{
  h->N = (int32_t)get_le(b + 16, 4); h->M = (int32_t)get_le(b + 20, 4); h->nh = (int32_t)get_le(b + 24, 4); h->mode = (int32_t)get_le(b + 28, 4);
  h->fingerprint = get_le(b + 32, 8);
  h->seed = (uint32_t)get_le(b + 40, 4); h->sweeps_per_call = (int32_t)get_le(b + 44, 4); h->manycd = (int32_t)get_le(b + 48, 4);
  h->store = (int32_t)get_le(b + 52, 4); h->max_samples = (int32_t)get_le(b + 56, 4); h->acc = (int32_t)get_le(b + 60, 4);
  h->calls_done = (int64_t)get_le(b + 64, 8);
  h->n_samples = (int32_t)get_le(b + 72, 4); h->sample_base = (int32_t)get_le(b + 76, 4); h->rows = (int32_t)get_le(b + 80, 4);
  h->n_chains = (int32_t)get_le(b + 84, 4);
  h->record_size = get_le(b + 88, 8);
}

/* Byte offsets of a record's parts.  The scalars (SER_CKPT_SCALARS bytes):
 *   0 f64 c, cc, d, dd, loglik, sum_negll, sum_ec, sum_ed | 64 i64 cursor | 72 i64 counters[8] | 136 i32 t0a, f0a, t1a, f1a |
 *   152 u32 sweep | 156 i32 n_samples | 160 u32 flags (bit 0: replay tape exhausted) | 164 u32 zero
 * then the parts below, each present only when the run has it, widest elements first so that every field is aligned. */
struct CkptLayout {
  long long cd;      /* f64 [4][M] c, log(1-e^c), d, log(1-e^d) per taxon (manycd)                */
  long long cdl;     /* f64 [rows][3] c, d, loglik of every stored row (SER_STORE_FULL)           */
  long long cd_all;  /* f64 [rows][2][M] per-taxon c, d of every stored row (FULL + manycd)       */
  long long acc;     /* i32 [acc_layout().ints] the chain's accumulator record (SER_ACC_*), up to rpi */
  long long rpi;     /* u16 [N] site at each position                                             */
  long long ab;      /* u16 [M] a, then u16 [M] b, per taxon                                       */
  long long spi;     /* u16 [rows][N] stored pi rows (SER_STORE_PI)                                */
  long long sa, sb;  /* u16 [rows][M] stored a, b rows (SER_STORE_FULL)                            */
  long long end;     /* end of the data; zero padding up to the checksum                          */
  long long size;    /* record bytes, checksum included                                           */
  int rows;
};

__host__ __device__ inline CkptLayout ckpt_layout(int N, int M, int manycd, int store, int rows, int acc)
{
  CkptLayout L;
  const long long n = N, m = M, r = rows;
  const bool full = store >= SER_STORE_FULL;
  long long o = SER_CKPT_SCALARS;
  L.rows = rows;
  L.cd = o; o += manycd ? 8 * 4 * m : 0;
  L.cdl = o; o += full ? 8 * 3 * r : 0;
  L.cd_all = o; o += (full && manycd) ? 8 * 2 * m * r : 0;
  L.acc = o; o += 4 * (long long)acc_layout(N, M, manycd, acc).ints;
  L.rpi = o; o += 2 * n;
  L.ab = o; o += 4 * m;
  L.spi = o; o += store >= SER_STORE_PI ? 2 * n * r : 0;
  L.sa = o; o += full ? 2 * m * r : 0;
  L.sb = o; o += full ? 2 * m * r : 0;
  L.end = o;
  L.size = (o + 7) / 8 * 8 + 8;
  return L;
}

/* dst[0, total) = src[0, valid), then zeros: rows past a chain's own count (a replay chain whose tape ran out) are written as
 * zeros so that a file never holds uninitialised bytes */
template <typename T>
__device__ __forceinline__ void ckpt_copy(T *dst, const T *src, long long valid, long long total)
{
  for (long long i = threadIdx.x; i < total; i += blockDim.x) dst[i] = i < valid ? src[i] : (T)0;
}

/* one record per block: local chain locals[blockIdx.x] into out + blockIdx.x * L.size (the checksum slot is left zero) */
__global__ void ser_ckpt_pack_kernel(KParams p, CkptLayout L, const int *acc, const int *locals, unsigned char *out)
{
  const int chain = locals[blockIdx.x], tid = threadIdx.x, nt = blockDim.x, N = p.N, M = p.M;
  unsigned char *rec = out + (size_t)blockIdx.x * L.size;
  const ChainScalars *sc = p.scal + chain;
  if (tid == 0) {
    double *f = (double *)rec;
    f[0] = sc->c; f[1] = sc->cc; f[2] = sc->d; f[3] = sc->dd; f[4] = sc->loglik; f[5] = sc->sum_negll; f[6] = sc->sum_ec; f[7] = sc->sum_ed;
    long long *q = (long long *)(rec + 64);
    q[0] = sc->cursor;
    for (int k = 0; k < 8; k++) q[1 + k] = sc->counters[k];
    int *i = (int *)(rec + 136);
    i[0] = sc->t0a; i[1] = sc->f0a; i[2] = sc->t1a; i[3] = sc->f1a;
    i[4] = (int)sc->sweep; i[5] = sc->n_samples; i[6] = sc->flags & 1; i[7] = 0;
  }
  uint16_t *rpi = (uint16_t *)(rec + L.rpi), *a = (uint16_t *)(rec + L.ab), *b = a + M;
  for (int n = tid; n < N; n += nt) rpi[n] = p.rpi[(size_t)chain * p.Npad + n];
  for (int c = tid; c < M; c += nt) { /* sorted column c holds taxon order[c] */
    const int tx = p.order[c];
    a[tx] = p.ab[(size_t)chain * 2 * p.Mpad + c];
    b[tx] = p.ab[(size_t)chain * 2 * p.Mpad + p.Mpad + c];
  }
  if (p.manycd) {
    double *cd = (double *)(rec + L.cd);
    for (int q = tid; q < 4 * M; q += nt) {
      const int k = q / M, c = q - k * M;
      cd[(size_t)k * M + p.order[c]] = p.cd4[(size_t)chain * 4 * p.Mpad + (size_t)k * p.Mpad + c];
    }
  }
  if (L.rows > 0) {
    const long long own = max(0, min(sc->n_samples - p.sample_base, L.rows)), row0 = (long long)chain * p.max_samples, R = L.rows;
    ckpt_copy((uint16_t *)(rec + L.spi), p.samp_pi + row0 * N, own * N, R * N);
    if (p.store >= SER_STORE_FULL) {
      ckpt_copy((uint16_t *)(rec + L.sa), p.samp_a + row0 * M, own * M, R * M);
      ckpt_copy((uint16_t *)(rec + L.sb), p.samp_b + row0 * M, own * M, R * M);
      ckpt_copy((double *)(rec + L.cdl), p.samp_cdl + row0 * 3, own * 3, R * 3);
      if (p.manycd) ckpt_copy((double *)(rec + L.cd_all), p.samp_cd_all + row0 * 2 * M, own * 2 * M, R * 2 * M);
    }
  }
  const long long na = (L.rpi - L.acc) / 4;
  if (acc) ckpt_copy((int *)(rec + L.acc), acc + chain * na, na, na);
  for (long long o = L.end + tid; o < L.size; o += nt) rec[o] = 0;
}

/* the mirror: record blockIdx.x of `in` into local chain locals[blockIdx.x].  The flags keep bit 0 alone: the bit columns
 * (SER_FLAG_COLUMNS) are rebuilt from rpi by the next sweep, and bits 1-4 are ser_check_kernel's to set. */
__global__ void ser_ckpt_unpack_kernel(KParams p, CkptLayout L, int *acc, const int *locals, const unsigned char *in)
{
  const int chain = locals[blockIdx.x], tid = threadIdx.x, nt = blockDim.x, N = p.N, M = p.M;
  const unsigned char *rec = in + (size_t)blockIdx.x * L.size;
  if (tid == 0) {
    ChainScalars sc;
    memset(&sc, 0, sizeof(sc));
    const double *f = (const double *)rec;
    sc.c = f[0]; sc.cc = f[1]; sc.d = f[2]; sc.dd = f[3]; sc.loglik = f[4]; sc.sum_negll = f[5]; sc.sum_ec = f[6]; sc.sum_ed = f[7];
    const long long *q = (const long long *)(rec + 64);
    sc.cursor = q[0];
    for (int k = 0; k < 8; k++) sc.counters[k] = q[1 + k];
    const int *i = (const int *)(rec + 136);
    sc.t0a = i[0]; sc.f0a = i[1]; sc.t1a = i[2]; sc.f1a = i[3];
    sc.sweep = (unsigned int)i[4]; sc.n_samples = i[5]; sc.flags = i[6] & 1;
    p.scal[chain] = sc;
  }
  const uint16_t *rpi = (const uint16_t *)(rec + L.rpi), *a = (const uint16_t *)(rec + L.ab), *b = a + M;
  for (int n = tid; n < N; n += nt) p.rpi[(size_t)chain * p.Npad + n] = rpi[n];
  for (int c = tid; c < M; c += nt) {
    const int tx = p.order[c];
    p.ab[(size_t)chain * 2 * p.Mpad + c] = a[tx];
    p.ab[(size_t)chain * 2 * p.Mpad + p.Mpad + c] = b[tx];
  }
  if (p.manycd) {
    const double *cd = (const double *)(rec + L.cd);
    for (int q = tid; q < 4 * M; q += nt) {
      const int k = q / M, c = q - k * M;
      p.cd4[(size_t)chain * 4 * p.Mpad + (size_t)k * p.Mpad + c] = cd[(size_t)k * M + p.order[c]];
    }
  }
  if (L.rows > 0) {
    const long long row0 = (long long)chain * p.max_samples, R = L.rows;
    ckpt_copy(p.samp_pi + row0 * N, (const uint16_t *)(rec + L.spi), R * N, R * N);
    if (p.store >= SER_STORE_FULL) {
      ckpt_copy(p.samp_a + row0 * M, (const uint16_t *)(rec + L.sa), R * M, R * M);
      ckpt_copy(p.samp_b + row0 * M, (const uint16_t *)(rec + L.sb), R * M, R * M);
      ckpt_copy(p.samp_cdl + row0 * 3, (const double *)(rec + L.cdl), R * 3, R * 3);
      if (p.manycd) ckpt_copy(p.samp_cd_all + row0 * 2 * M, (const double *)(rec + L.cd_all), R * 2 * M, R * 2 * M);
    }
  }
  const long long na = (L.rpi - L.acc) / 4;
  if (acc) ckpt_copy(acc + chain * na, (const int *)(rec + L.acc), na, na);
}

/* ------------------------------------------------------------------ host side */
static int run_global_id(const ser_run *run, int c) { return run->h_chain_ids ? run->h_chain_ids[c] : run->cfg.chain_offset + c; }

/* stored rows per chain: a store keeps the samples taken since sample_base, at most max_samples of them */
static int ckpt_rows(int store, int max_samples, int n_samples, int sample_base)
{
  if (store < SER_STORE_PI) return 0;
  return std::max(0, std::min(n_samples - sample_base, max_samples));
}

static CkptLayout ckpt_layout_of(const CkptHeader &h) { return ckpt_layout(h.N, h.M, h.manycd, h.store, h.rows, h.acc); }

static long long ckpt_table_bytes(int n) { return ((long long)n * 4 + 7) / 8 * 8 + 8; }

static int write_all(int fd, const void *buf, size_t n, off_t off)
{
  const char *p = (const char *)buf;
  while (n > 0) {
    const ssize_t w = pwrite(fd, p, n, off);
    if (w < 0 && errno == EINTR) continue;
    if (w <= 0) return -1;
    p += w; n -= (size_t)w; off += w;
  }
  return 0;
}

static int read_all(int fd, void *buf, size_t n, off_t off)
{
  char *p = (char *)buf;
  while (n > 0) {
    const ssize_t r = pread(fd, p, n, off);
    if (r < 0 && errno == EINTR) continue;
    if (r <= 0) return -1;
    p += r; n -= (size_t)r; off += r;
  }
  return 0;
}

/* Header (and, with `table`, the chain table) of an open checkpoint, validated: magic, version, checksums, a layout that
 * matches the record size, and a file exactly as long as header + table + records.  *data_off = first record. */
static int ckpt_read_head(int fd, const char *path, CkptHeader *h, std::vector<int> *table, long long *data_off)
{
  unsigned char b[SER_CKPT_HEADER];
  struct stat st;
  if (fstat(fd, &st) != 0) { ser_set_error("checkpoint %s: %s", path, strerror(errno)); return SER_E_IO; }
  if (st.st_size < SER_CKPT_HEADER || read_all(fd, b, SER_CKPT_HEADER, 0)) { ser_set_error("checkpoint %s: truncated header", path); return SER_E_IO; }
  if (memcmp(b, "SERCKPT", 8)) { ser_set_error("checkpoint %s: bad magic (not a checkpoint file)", path); return SER_E_IO; }
  if (get_le(b + 8, 4) != SER_CKPT_VERSION || get_le(b + 12, 4) != SER_CKPT_HEADER) {
    ser_set_error("checkpoint %s: format version %u with a %u-byte header; this library reads version %u", path, (unsigned)get_le(b + 8, 4),
                  (unsigned)get_le(b + 12, 4), SER_CKPT_VERSION);
    return SER_E_IO;
  }
  if (get_le(b + 96, 8) != ckpt_hash(b, 96)) { ser_set_error("checkpoint %s: header checksum mismatch", path); return SER_E_IO; }
  ckpt_decode_header(b, h);
  const bool sane = h->N >= 2 && h->N <= SER_MAX_SITES && h->M >= 1 && h->M <= SER_MAX_TAXA && h->n_chains >= 1 && h->max_samples >= 0 &&
                    h->store >= SER_STORE_NONE && h->store <= SER_STORE_FULL && (h->manycd == 0 || h->manycd == 1) && h->n_samples >= 0 &&
                    h->sample_base >= 0 && h->sample_base <= h->n_samples && h->calls_done >= h->n_samples &&
                    h->rows == ckpt_rows(h->store, h->max_samples, h->n_samples, h->sample_base) && (h->acc & ~SER_ACC_ALL) == 0;
  if (!sane) { ser_set_error("checkpoint %s: inconsistent header fields", path); return SER_E_IO; }
  if (h->record_size != (uint64_t)ckpt_layout_of(*h).size) {
    ser_set_error("checkpoint %s: record size %llu does not match the layout of its header (%lld)", path, (unsigned long long)h->record_size,
                  ckpt_layout_of(*h).size);
    return SER_E_IO;
  }
  const long long doff = SER_CKPT_HEADER + ckpt_table_bytes(h->n_chains);
  const long long rs = (long long)h->record_size, body = (long long)st.st_size - doff;
  if (body < 0 || body % rs != 0 || body / rs != h->n_chains) {
    ser_set_error("checkpoint %s: %lld bytes, the header describes %lld (truncated or extended file)", path, (long long)st.st_size,
                  doff + (long long)h->n_chains * (long long)h->record_size);
    return SER_E_IO;
  }
  if (data_off) *data_off = doff;
  if (table) {
    std::vector<unsigned char> t((size_t)ckpt_table_bytes(h->n_chains));
    if (read_all(fd, t.data(), t.size(), SER_CKPT_HEADER)) { ser_set_error("checkpoint %s: cannot read the chain table", path); return SER_E_IO; }
    if (get_le(t.data() + t.size() - 8, 8) != ckpt_hash(t.data(), t.size() - 8)) { ser_set_error("checkpoint %s: chain table checksum mismatch", path); return SER_E_IO; }
    table->resize(h->n_chains);
    for (int i = 0; i < h->n_chains; i++) {
      (*table)[i] = (int32_t)get_le(t.data() + 4 * i, 4);
      if ((*table)[i] < 0 || (i && (*table)[i] <= (*table)[i - 1])) { ser_set_error("checkpoint %s: chain table not ascending at entry %d", path, i); return SER_E_IO; }
    }
  }
  return SER_OK;
}

/* pinned staging of at most SER_CKPT_STAGING bytes (one record at least) and its device twin on the run's device */
struct CkptStage {
  unsigned char *host = nullptr;
  size_t bytes = 0;
  int per_block = 0;
  ~CkptStage() { if (host) cudaFreeHost(host); }
  int alloc(long long rec_size, long long n_records)
  {
    per_block = (int)std::max<long long>(1, std::min<long long>(n_records, (long long)(SER_CKPT_STAGING / (unsigned long long)rec_size)));
    bytes = (size_t)per_block * (size_t)rec_size;
    CUDA_TRY(cudaMallocHost((void **)&host, bytes));
    return SER_OK;
  }
};

static void ckpt_header_of(const ser_run *run, int n_chains, CkptHeader *h)
{
  memset(h, 0, sizeof(*h));
  h->N = run->N; h->M = run->M; h->nh = run->nh; h->mode = run->cfg.mode; h->fingerprint = run->ds_fp;
  h->seed = run->cfg.seed; h->sweeps_per_call = run->cfg.sweeps_per_call; h->manycd = run->cfg.manycd; h->store = run->cfg.store;
  h->max_samples = run->cfg.max_samples; h->acc = run->acc_what;
  h->calls_done = run->calls_done; h->n_samples = run->samples_done; h->sample_base = run->kp.sample_base;
  h->rows = ckpt_rows(h->store, h->max_samples, h->n_samples, h->sample_base);
  h->n_chains = n_chains;
  h->record_size = (uint64_t)ckpt_layout_of(*h).size;
}

/* The chains of `runs` (one run, or the devices of a ser_multi) into one file in ascending global id: path.tmp is written,
 * flushed and synced, then renamed over path, so a crash mid-write leaves the previous file intact. */
static int ckpt_save(ser_run *const *runs, int n_runs, const char *path, const char *who)
{
  if (!path) { ser_set_error("%s: null path", who); return SER_E_ARG; }
  struct Ref { int g, r, c; };
  std::vector<Ref> refs;
  for (int r = 0; r < n_runs; r++) {
    ser_run *run = runs[r];
    if (!run->initialized) { ser_set_error("%s: the run is not initialised (ser_run_init or a checkpoint load first)", who); return SER_E_STATE; }
    if (set_device(run)) return SER_E_CUDA;
    CUDA_TRY(cudaStreamSynchronize(run->stream));
    for (int c = 0; c < run->cfg.n_chains; c++) refs.push_back(Ref{run_global_id(run, c), r, c});
  }
  std::sort(refs.begin(), refs.end(), [](const Ref &x, const Ref &y) { return x.g < y.g; });
  CkptHeader h;
  ckpt_header_of(runs[0], (int)refs.size(), &h);
  const CkptLayout L = ckpt_layout_of(h);
  const long long doff = SER_CKPT_HEADER + ckpt_table_bytes(h.n_chains);
  std::vector<unsigned char> head((size_t)doff, 0);
  ckpt_encode_header(h, head.data());
  for (size_t i = 0; i < refs.size(); i++) put_le(head.data() + SER_CKPT_HEADER + 4 * i, (uint32_t)refs[i].g, 4);
  put_le(head.data() + doff - 8, ckpt_hash(head.data() + SER_CKPT_HEADER, (size_t)(doff - 8 - SER_CKPT_HEADER)), 8);

  const std::string tmp = std::string(path) + ".tmp";
  const int fd = open(tmp.c_str(), O_WRONLY | O_CREAT | O_TRUNC | O_CLOEXEC, 0644);
  if (fd < 0) { ser_set_error("%s: cannot create %s: %s", who, tmp.c_str(), strerror(errno)); return SER_E_IO; }
  CkptStage stage;
  auto body = [&]() -> int {
    if (write_all(fd, head.data(), head.size(), 0)) { ser_set_error("%s: cannot write %s: %s", who, tmp.c_str(), strerror(errno)); return SER_E_IO; }
    int rc = stage.alloc(L.size, h.n_chains);
    if (rc) return rc;
    for (int r = 0; r < n_runs; r++) {
      ser_run *run = runs[r];
      std::vector<int> pos, loc; /* this run's chains in file order: position in the table, local index */
      for (size_t i = 0; i < refs.size(); i++) if (refs[i].r == r) { pos.push_back((int)i); loc.push_back(refs[i].c); }
      if (set_device(run)) return SER_E_CUDA;
      unsigned char *d_stage = nullptr;
      int *d_loc = nullptr;
      auto per_run = [&]() -> int {
        CUDA_TRY(POOL_ALLOC(&d_stage, stage.bytes));
        CUDA_TRY(POOL_ALLOC(&d_loc, (size_t)stage.per_block * sizeof(int)));
        for (size_t i0 = 0; i0 < pos.size(); i0 += stage.per_block) {
          const int nb = (int)std::min<size_t>(stage.per_block, pos.size() - i0);
          CUDA_TRY(cudaMemcpyAsync(d_loc, loc.data() + i0, (size_t)nb * sizeof(int), cudaMemcpyHostToDevice, run->stream));
          mark_launch(run);
          ser_ckpt_pack_kernel<<<nb, 256, 0, run->stream>>>(run->kp, L, run->d_acc, d_loc, d_stage);
          CUDA_TRY(cudaGetLastError());
          CUDA_TRY(cudaMemcpyAsync(stage.host, d_stage, (size_t)nb * L.size, cudaMemcpyDeviceToHost, run->stream));
          CUDA_TRY(cudaStreamSynchronize(run->stream));
          for (int j = 0; j < nb; j++) {
            unsigned char *rec = stage.host + (size_t)j * L.size;
            put_le(rec + L.size - 8, ckpt_hash(rec, (size_t)L.size - 8), 8);
          }
          for (int j = 0; j < nb;) { /* runs of consecutive table positions go out in one write */
            int k = j + 1;
            while (k < nb && pos[i0 + k] == pos[i0 + k - 1] + 1) k++;
            if (write_all(fd, stage.host + (size_t)j * L.size, (size_t)(k - j) * L.size, (off_t)(doff + (long long)pos[i0 + j] * L.size))) {
              ser_set_error("%s: cannot write %s: %s", who, tmp.c_str(), strerror(errno));
              return SER_E_IO;
            }
            j = k;
          }
        }
        return SER_OK;
      };
      rc = per_run();
      if (d_stage) cudaFreeAsync(d_stage, run->stream);
      if (d_loc) cudaFreeAsync(d_loc, run->stream);
      if (rc) return rc;
    }
    if (fsync(fd) != 0) { ser_set_error("%s: fsync %s: %s", who, tmp.c_str(), strerror(errno)); return SER_E_IO; }
    return SER_OK;
  };
  int rc = body();
  if (close(fd) != 0 && rc == SER_OK) { ser_set_error("%s: close %s: %s", who, tmp.c_str(), strerror(errno)); rc = SER_E_IO; }
  if (rc == SER_OK && rename(tmp.c_str(), path) != 0) { ser_set_error("%s: rename %s -> %s: %s", who, tmp.c_str(), path, strerror(errno)); rc = SER_E_IO; }
  if (rc != SER_OK) unlink(tmp.c_str());
  return rc;
}

/* One permutation row (u16 [N] at perm) and, with ab, one a/b row (u16 [M] a at ab, u16 [M] b at ab + b_off) of chain g: the
 * permutation holds each of 0..N-1 once, and every taxon has a <= b <= N.  `row` < 0 names the live state, else a stored row. */
static int ckpt_check_rows(const unsigned char *perm, const char *perm_name, const unsigned char *ab, long long b_off, const char *ab_name,
                           int N, int M, std::vector<unsigned char> &seen, int g, long long row, const char *who)
{
  char where[40] = "";
  auto name_row = [&]() { if (row >= 0) snprintf(where, sizeof(where), "stored row %lld: ", row); };
  std::fill(seen.begin(), seen.end(), 0);
  for (int n = 0; n < N; n++) {
    const int s = (int)get_le(perm + 2 * n, 2);
    if (s >= N || seen[s]) {
      name_row();
      ser_set_error("%s: chain %d: %s%s is not a permutation of 0..%d (entry %d holds %d)", who, g, where, perm_name, N - 1, n, s);
      return SER_E_CHECK;
    }
    seen[s] = 1;
  }
  if (ab)
    for (int m = 0; m < M; m++) {
      const int a = (int)get_le(ab + 2 * m, 2), b = (int)get_le(ab + b_off + 2 * m, 2);
      if (!(a <= b && b <= N)) {
        name_row();
        ser_set_error("%s: chain %d: %s%s of taxon %d has a = %d, b = %d (needs a <= b <= %d)", who, g, where, ab_name, m, a, b, N);
        return SER_E_CHECK;
      }
    }
  return SER_OK;
}

/* What a record may hold before it goes near a kernel.  The sweep kernels index shared memory with rpi and a/b, the tape with
 * the cursor and the sample store with n_samples - sample_base.  The histogram kernels (ser_run_marginals and the SER_ACC_POS /
 * SER_ACC_RANGE accumulators) index their rows with the stored pi, a and b, so the chain's own stored rows obey the rules of the
 * state; rows past its own count are never read and stay unchecked.  Checked on the host, from the file's bytes. */
static int ckpt_check_record(const unsigned char *rec, const CkptLayout &L, const CkptHeader &h, long long tape_len, int g, const char *who)
{
  const int N = h.N, M = h.M;
  const long long cursor = (long long)get_le(rec + 64, 8);
  const int n_samples = (int32_t)get_le(rec + 156, 4);
  const uint32_t flags = (uint32_t)get_le(rec + 160, 4);
  if (flags > 1) { ser_set_error("%s: chain %d: flags %u (only bit 0, tape exhausted, is stored)", who, g, flags); return SER_E_CHECK; }
  std::vector<unsigned char> seen(N);
  int rc = ckpt_check_rows(rec + L.rpi, "rpi", rec + L.ab, 2ll * M, "a/b", N, M, seen, g, -1, who);
  if (rc) return rc;
  if (cursor < 0) { ser_set_error("%s: chain %d: negative tape cursor %lld", who, g, cursor); return SER_E_CHECK; }
  if (!(flags & 1) && h.mode == SER_MODE_REPLAY && cursor > tape_len) { /* a chain whose tape ran out never sweeps again */
    ser_set_error("%s: chain %d: replay cursor %lld is beyond its tape of %lld draws", who, g, cursor, tape_len);
    return SER_E_TAPE;
  }
  /* an exhausted chain may hold fewer samples than sample_base, never more than the run: the reductions read
   * min(n_samples, max_samples) of its rows */
  if (n_samples > h.n_samples || (!(flags & 1) && n_samples < h.sample_base)) {
    ser_set_error("%s: chain %d: n_samples %d outside [sample_base %d, %d]", who, g, n_samples, h.sample_base, h.n_samples);
    return SER_E_CHECK;
  }
  const bool full = h.store >= SER_STORE_FULL;
  const long long own = std::max(0ll, std::min((long long)n_samples - h.sample_base, (long long)L.rows));
  for (long long t = 0; t < own; t++) {
    rc = ckpt_check_rows(rec + L.spi + 2 * N * t, "spi", full ? rec + L.sa + 2 * M * t : nullptr, L.sb - L.sa, "sa/sb", N, M, seen, g, t, who);
    if (rc) return rc;
  }
  return SER_OK;
}

/* the run's side of a load: look up its chains, range-check and upload their records block by block, rebuild what ser_run_init
 * sets, then ser_check_kernel over the run */
static int ckpt_load_run(ser_run *run, int fd, const char *path, const CkptHeader &h, const std::vector<int> &table, long long doff,
                         CkptStage &stage, const char *who)
{
  const int nc = run->cfg.n_chains;
  const CkptLayout L = ckpt_layout_of(h);
  std::vector<std::pair<int, int>> pl(nc); /* (position in the file, local chain) */
  for (int c = 0; c < nc; c++) {
    const int g = run_global_id(run, c);
    const auto it = std::lower_bound(table.begin(), table.end(), g);
    if (it == table.end() || *it != g) { ser_set_error("%s: chain %d is not in %s", who, g, path); return SER_E_ARG; }
    pl[c] = std::make_pair((int)(it - table.begin()), c);
  }
  std::sort(pl.begin(), pl.end());
  if (set_device(run)) return SER_E_CUDA;
  std::vector<unsigned long long> toff;
  if (h.mode == SER_MODE_REPLAY) {
    toff.resize((size_t)nc + 1);
    CUDA_TRY(cudaMemcpyAsync(toff.data(), run->d_tape_off, toff.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, run->stream));
  }
  CUDA_TRY(cudaStreamSynchronize(run->stream));
  unsigned char *d_stage = nullptr;
  int *d_loc = nullptr;
  std::vector<int> loc(stage.per_block);
  auto blocks = [&]() -> int {
    CUDA_TRY(POOL_ALLOC(&d_stage, stage.bytes));
    CUDA_TRY(POOL_ALLOC(&d_loc, (size_t)stage.per_block * sizeof(int)));
    for (int i0 = 0; i0 < nc; i0 += stage.per_block) {
      const int nb = std::min(stage.per_block, nc - i0);
      for (int j = 0; j < nb;) {
        int k = j + 1;
        while (k < nb && pl[i0 + k].first == pl[i0 + k - 1].first + 1) k++;
        if (read_all(fd, stage.host + (size_t)j * L.size, (size_t)(k - j) * L.size, (off_t)(doff + (long long)pl[i0 + j].first * L.size))) {
          ser_set_error("%s: %s: cannot read records: %s", who, path, strerror(errno));
          return SER_E_IO;
        }
        j = k;
      }
      for (int j = 0; j < nb; j++) {
        const unsigned char *rec = stage.host + (size_t)j * L.size;
        const int c = pl[i0 + j].second, g = table[pl[i0 + j].first];
        if (get_le(rec + L.size - 8, 8) != ckpt_hash(rec, (size_t)L.size - 8)) { ser_set_error("%s: %s: record of chain %d: checksum mismatch", who, path, g); return SER_E_IO; }
        const long long tape_len = toff.empty() ? 0 : (long long)(toff[c + 1] - toff[c]);
        const int rc = ckpt_check_record(rec, L, h, tape_len, g, who);
        if (rc) return rc;
        loc[j] = c;
      }
      CUDA_TRY(cudaMemcpyAsync(d_stage, stage.host, (size_t)nb * L.size, cudaMemcpyHostToDevice, run->stream));
      CUDA_TRY(cudaMemcpyAsync(d_loc, loc.data(), (size_t)nb * sizeof(int), cudaMemcpyHostToDevice, run->stream));
      mark_launch(run);
      ser_ckpt_unpack_kernel<<<nb, 256, 0, run->stream>>>(run->kp, L, run->d_acc, d_loc, d_stage);
      CUDA_TRY(cudaGetLastError());
      CUDA_TRY(cudaStreamSynchronize(run->stream)); /* the pinned buffer and loc are refilled by the next block */
    }
    return SER_OK;
  };
  int rc = blocks();
  if (d_stage) cudaFreeAsync(d_stage, run->stream);
  if (d_loc) cudaFreeAsync(d_loc, run->stream);
  if (rc) return rc;
  /* what ser_run_init sets, then the restored counters */
  if (run->d_done) CUDA_TRY(cudaMemsetAsync(run->d_done, 0, (size_t)nc * sizeof(unsigned int), run->stream));
  run->chunks_done = 0;
  run->kp.sample_base = h.sample_base;
  run->sampled = h.n_samples > 0;
  run->calls_done = h.calls_done;
  run->samples_done = h.n_samples;
  CUDA_TRY(cudaMemsetAsync(run->d_bad, 0, sizeof(int), run->stream));
  mark_launch(run);
  ser_check_kernel<<<nc, run->Caux, run->smem_small, run->stream>>>(run->kp, run->d_bad);
  CUDA_TRY(cudaGetLastError());
  std::vector<ChainScalars> sc(nc);
  CUDA_TRY(cudaMemcpyAsync(sc.data(), run->d_scal, (size_t)nc * sizeof(ChainScalars), cudaMemcpyDeviceToHost, run->stream));
  CUDA_TRY(cudaStreamSynchronize(run->stream));
  for (int c = 0; c < nc; c++)
    if (sc[c].flags & 30) { /* bit 0 (tape exhausted) is state, not an inconsistency */
      ser_set_error("%s: chain %d fails the consistency check (flags %d: 2 a/b range, 4 permutation, 8 hard-site order, 16 totals / log-likelihood)",
                    who, run_global_id(run, c), sc[c].flags & 30);
      return SER_E_CHECK;
    }
  run->initialized = 1;
  return SER_OK;
}

static int ckpt_load(ser_run *const *runs, int n_runs, const char *path, const char *who)
{
  for (int r = 0; r < n_runs; r++) runs[r]->initialized = 0; /* whatever fails below, no sweep runs on this state */
  if (!path) { ser_set_error("%s: null path", who); return SER_E_ARG; }
  const int fd = open(path, O_RDONLY | O_CLOEXEC);
  if (fd < 0) { ser_set_error("%s: cannot open %s: %s", who, path, strerror(errno)); return SER_E_IO; }
  CkptHeader h;
  std::vector<int> table;
  long long doff = 0;
  CkptStage stage;
  auto body = [&]() -> int {
    int rc = ckpt_read_head(fd, path, &h, &table, &doff);
    if (rc) return rc;
    for (int r = 0; r < n_runs; r++) {
      const ser_run *run = runs[r];
      if (h.N != run->N || h.M != run->M || h.nh != run->nh || h.fingerprint != run->ds_fp) {
        ser_set_error("%s: %s holds chains of another dataset (%d x %d, fingerprint %016llx; this run: %d x %d, %016llx)", who, path, h.N, h.M,
                      (unsigned long long)h.fingerprint, run->N, run->M, (unsigned long long)run->ds_fp);
        return SER_E_ARG;
      }
      const struct { const char *name; long long file, here; } cfg[] = {
          {"mode", h.mode, run->cfg.mode}, {"seed", h.seed, run->cfg.seed}, {"sweeps_per_call", h.sweeps_per_call, run->cfg.sweeps_per_call},
          {"manycd", h.manycd, run->cfg.manycd}, {"store", h.store, run->cfg.store}, {"max_samples", h.max_samples, run->cfg.max_samples},
          {"accumulate flags", h.acc, run->acc_what}};
      for (const auto &f : cfg)
        if (f.file != f.here) { ser_set_error("%s: %s was saved with %s = %lld, this run has %lld", who, path, f.name, f.file, f.here); return SER_E_STATE; }
      if (run->cfg.mode == SER_MODE_REPLAY && !run->have_tapes) { ser_set_error("%s: replay mode needs ser_run_set_tapes first", who); return SER_E_TAPE; }
    }
    int most = 1; /* a subset run stages no more than its own chains */
    for (int r = 0; r < n_runs; r++) most = std::max(most, runs[r]->cfg.n_chains);
    if ((rc = stage.alloc(h.record_size, std::min(most, h.n_chains)))) return rc;
    for (int r = 0; r < n_runs; r++)
      if ((rc = ckpt_load_run(runs[r], fd, path, h, table, doff, stage, who))) return rc;
    return SER_OK;
  };
  const int rc = body();
  close(fd);
  if (rc) for (int r = 0; r < n_runs; r++) runs[r]->initialized = 0;
  return rc;
}

/* ------------------------------------------------------------------ C ABI */
extern "C" int ser_run_save_checkpoint(ser_run *run, const char *path)
{
  if (!run) { ser_set_error("ser_run_save_checkpoint: null run"); return SER_E_ARG; }
  return ckpt_save(&run, 1, path, "ser_run_save_checkpoint");
}

extern "C" int ser_run_load_checkpoint(ser_run *run, const char *path)
{
  if (!run) { ser_set_error("ser_run_load_checkpoint: null run"); return SER_E_ARG; }
  return ckpt_load(&run, 1, path, "ser_run_load_checkpoint");
}

extern "C" int ser_multi_save_checkpoint(ser_multi *m, const char *path)
{
  if (!m) { ser_set_error("ser_multi_save_checkpoint: null argument"); return SER_E_ARG; }
  return ckpt_save(m->run, m->n_gpus, path, "ser_multi_save_checkpoint");
}

extern "C" int ser_multi_load_checkpoint(ser_multi *m, const char *path)
{
  if (!m) { ser_set_error("ser_multi_load_checkpoint: null argument"); return SER_E_ARG; }
  return ckpt_load(m->run, m->n_gpus, path, "ser_multi_load_checkpoint");
}

extern "C" int ser_checkpoint_info(const char *path, int32_t *N, int32_t *M, int32_t *n_chains, int64_t *calls_done, int32_t *n_samples,
                                   uint32_t *seed, int32_t *mode, int32_t *manycd)
{
  if (!path) { ser_set_error("ser_checkpoint_info: null path"); return SER_E_ARG; }
  const int fd = open(path, O_RDONLY | O_CLOEXEC);
  if (fd < 0) { ser_set_error("ser_checkpoint_info: cannot open %s: %s", path, strerror(errno)); return SER_E_IO; }
  CkptHeader h;
  const int rc = ckpt_read_head(fd, path, &h, nullptr, nullptr);
  close(fd);
  if (rc) return rc;
  if (N) *N = h.N;
  if (M) *M = h.M;
  if (n_chains) *n_chains = h.n_chains;
  if (calls_done) *calls_done = h.calls_done;
  if (n_samples) *n_samples = h.n_samples;
  if (seed) *seed = h.seed;
  if (mode) *mode = h.mode;
  if (manycd) *manycd = h.manycd;
  return SER_OK;
}
