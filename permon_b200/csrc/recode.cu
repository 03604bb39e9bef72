// Device re-coder: builds the stored form of a matrix whose CSR already lives in device memory, on the device.
//
// upload_csr (shim.cpp) turns a HOST CSR into the all-stencil form, packed dictionary tiles or padded CSR (pack.cpp).  A caller whose
// matrix is in HBM would otherwise copy it to the host first (12 B per non-zero over PCIe) and re-code it on the CPU.  The kernels here
// make the same decisions from the same statistics (spmv_stats / spmv_decide, pk_build's tile rules) and produce byte-identical arrays:
//   - row statistics: one reduction over the row pointer (longest row, most non-zeros of a 256-row tile);
//   - stencil tiles: one CTA per tile forms the union of its rows' (col - row, value bits) pairs in shared memory; the union is a set,
//     so the result does not depend on the order in which the threads insert;
//   - dictionary tiles: one CTA per tile hashes the (delta, value bits) pairs and ranks them by their FIRST storage index (atomicMin),
//     which is exactly the code order of the host's scan;
//   - layout: tile sizes -> prefix sum on the host (ntiles numbers) -> one fill kernel into a zeroed blob.
// Only per-tile scalars and the tiles where the stencil pattern changes are copied to the host.
#include <climits>
#include <cstring>
#include <algorithm>
#include <vector>

#include "objects.h"

namespace pb {

namespace {
constexpr int RT = 256;   // threads per CTA: one per row of a tile

// the pattern of a stencil tile: L (col - row, value bits) pairs, ascending delta; entries beyond L are zero
struct RcPat {
  int                t, L;
  int                d[8];
  unsigned long long b[8];
};

__device__ __forceinline__ unsigned long long dbits(double v) { return (unsigned long long)__double_as_longlong(v); }

// longest row and most non-zeros of a tile (spmv_stats)
__global__ void __launch_bounds__(RT) k_rc_stats(int n, const int *__restrict__ ia, int *out /* [0]: longest row, [1]: tile cap */)
{
  int mr = 0, cap = 0;
  for (int r = blockIdx.x * RT + threadIdx.x; r < n; r += gridDim.x * RT) {
    const int k = ia[r];
    mr = max(mr, ia[r + 1] - k);
    if ((r & (TR - 1)) == 0) cap = max(cap, ia[min(r + TR, n)] - k);
  }
  for (int o = 16; o; o >>= 1) {
    mr  = max(mr, __shfl_xor_sync(0xffffffffu, mr, o));
    cap = max(cap, __shfl_xor_sync(0xffffffffu, cap, o));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMax(out, mr);
    atomicMax(out + 1, cap);
  }
}

// longest row of every tile (tile-ELL widths)
__global__ void __launch_bounds__(RT) k_rc_tile_maxrow(int n, const int *__restrict__ ia, int *__restrict__ lt)
{
  __shared__ int m;
  if (threadIdx.x == 0) m = 0;
  __syncthreads();
  const int r = blockIdx.x * TR + threadIdx.x;
  if (r < n) atomicMax(&m, ia[r + 1] - ia[r]);
  __syncthreads();
  if (threadIdx.x == 0) lt[blockIdx.x] = m;
}

// stencil test of one tile (pk_build): every row sorted by column, every delta with one value, at most 8 distinct deltas, tile not
// empty.  Only the entries with a column in [c0, c1) take part, with local column col - c0 (the diagonal block of a row-partitioned
// matrix, pk_stencil_windowed; one rank passes the whole column range).  Writes the presence byte of every row of the tile (zero past
// n), the pattern, the tile's kind / header / blob size, and adds the tile's entries in the window to *nwin_nnz.
// The first thread that claims a delta's slot stores its value; every entry is compared with it after the barrier, so the verdict does
// not depend on which thread claimed first.
__global__ void __launch_bounds__(RT) k_rc_stencil(int n, const int *__restrict__ ia, const int *__restrict__ ja, const double *__restrict__ a, int c0,
                                                   int c1, unsigned char *__restrict__ masks, RcPat *__restrict__ tpat, unsigned char *__restrict__ tkind,
                                                   PkHeader *__restrict__ thdr, unsigned *__restrict__ tbytes, unsigned *nst, unsigned long long *nwin_nnz)
{
  __shared__ int                key[64];
  __shared__ unsigned long long vb[64];
  __shared__ int                bad, pd[8], tile_nnz;
  __shared__ unsigned long long pb[8];
  const int t = blockIdx.x, r0 = t * TR, r1 = min(r0 + TR, n), r = r0 + threadIdx.x;
  if (threadIdx.x < 64) key[threadIdx.x] = INT_MIN;   // col - row of columns and rows below 2^31 is never INT_MIN
  if (threadIdx.x == 0) bad = tile_nnz = 0;
  __syncthreads();
  volatile int *vkey = key;
  int           mine = 0;
  if (r < r1) {
    int prev = 0;
    for (int k = ia[r]; k < ia[r + 1]; k++) {
      const int c = ja[k];
      if (c < c0 || c >= c1) continue;   // ghost column
      const int d = c - c0 - r;
      if (mine && d <= prev) {
        bad = 1;
        break;
      }
      prev = d;
      mine++;
      unsigned h = ((unsigned)d * 0x9E3779B1u) >> 26, p = 0;
      for (; p < 64; p++, h = (h + 1) & 63) {
        const int cur = vkey[h];
        if (cur == d) break;
        if (cur == INT_MIN) {
          const int old = atomicCAS(&key[h], INT_MIN, d);
          if (old == INT_MIN) {
            vb[h] = dbits(a[k]);
            break;
          }
          if (old == d) break;
        }
      }
      if (p == 64) {   // more than 64 distinct deltas
        bad = 1;
        break;
      }
    }
  }
  if (mine) atomicAdd(&tile_nnz, mine);
  __syncthreads();
  const bool occ  = threadIdx.x < 64 && key[threadIdx.x] != INT_MIN;
  const int  nocc = __syncthreads_count(occ);
  if (occ) {
    int rank = 0;
    for (int q = 0; q < 64; q++) rank += (key[q] != INT_MIN && key[q] < key[threadIdx.x]);
    if (rank < 8) {
      pd[rank] = key[threadIdx.x];
      pb[rank] = vb[threadIdx.x];
    }
  }
  __syncthreads();
  bool fail = bad || nocc > 8 || tile_nnz == 0;
  unsigned m = 0;
  if (!fail && r < r1) {   // presence bits against the final pattern; an entry whose value differs from its delta's rejects the tile
    int j = 0;
    for (int k = ia[r]; k < ia[r + 1]; k++) {
      const int c = ja[k];
      if (c < c0 || c >= c1) continue;
      const int d = c - c0 - r;
      while (pd[j] != d) j++;
      if (dbits(a[k]) != pb[j]) bad = 1;
      m |= 1u << j;
      j++;
    }
  }
  __syncthreads();
  if (fail || bad) {
    if (threadIdx.x == 0) {
      tkind[t]  = 0xFF;
      tpat[t].L = 0;
    }
    return;
  }
  const int L = nocc;
  masks[(size_t)t * TR + threadIdx.x] = (unsigned char)m;
  if (threadIdx.x == 0) {
    RcPat P;
    P.t = t;
    P.L = L;
    for (int j = 0; j < 8; j++) {
      P.d[j] = j < L ? pd[j] : 0;
      P.b[j] = j < L ? pb[j] : 0ull;
    }
    tpat[t]  = P;
    tkind[t] = 2;
    PkHeader H;
    H.kind    = 2;
    H.ndict   = (uint16_t)L;
    H.nnz     = (uint32_t)(ia[r1] - ia[r0]);
    H.ulen    = (uint16_t)L;
    H.nrows   = (uint16_t)(r1 - r0);
    H.pad     = 0;
    thdr[t]   = H;
    tbytes[t] = (unsigned)pk_stencil_bytes(L, r1 - r0);
    atomicAdd(nst, 1u);
    atomicAdd(nwin_nnz, (unsigned long long)tile_nnz);
  }
}

__device__ __forceinline__ bool rc_pat_eq(const RcPat &x, const RcPat &y)
{
  if (x.L != y.L) return false;
  for (int j = 0; j < x.L; j++)
    if (x.d[j] != y.d[j] || x.b[j] != y.b[j]) return false;
  return true;
}

// tiles whose pattern differs from the previous tile's (the slot order follows atomics; the host sorts the records by tile)
__global__ void k_rc_changes(int ntiles, const RcPat *__restrict__ tpat, RcPat *__restrict__ rec, unsigned *cnt)
{
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < ntiles; t += gridDim.x * blockDim.x)
    if (t == 0 || !rc_pat_eq(tpat[t], tpat[t - 1])) rec[atomicAdd(cnt, 1u)] = tpat[t];
}

// pattern id of every tile: the id of the last run that starts at or before it
__global__ void k_rc_fill_pid(int ntiles, int nruns, const int *__restrict__ run_t, const unsigned char *__restrict__ run_id, unsigned char *__restrict__ pid)
{
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < ntiles; t += gridDim.x * blockDim.x) {
    int lo = 0, hi = nruns - 1;   // run_t[0] == 0
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (run_t[mid] <= t) lo = mid;
      else hi = mid - 1;
    }
    pid[t] = run_id[lo];
  }
}

constexpr int DS = 2048;   // hash slots of a tile dictionary (at most 512 keys are ever inserted: 256 + one per thread)

__device__ __forceinline__ unsigned rc_hash(int d, unsigned long long b)
{
  const unsigned long long h = (b ^ (b >> 29)) * 0x9E3779B97F4A7C15ull + (unsigned long long)(unsigned)d * 0xC2B2AE3D27D4EB4Full;
  return (unsigned)(h >> 40) & (DS - 1);
}
__device__ __forceinline__ int rc_row_of(const int *sia, int nrows, int k)   // last row whose first entry is <= k
{
  int lo = 0, hi = nrows - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (sia[mid] <= k) lo = mid;
    else hi = mid - 1;
  }
  return lo;
}

// dictionary of one non-stencil tile (pk_build's TileDict): the distinct (delta, value bits) pairs, coded in the order of their first
// occurrence in storage order; more than 256 pairs make a raw tile.  Writes one code byte per non-zero into `codes` and the tile's
// header and blob size (uniform rows, padded short ragged rows or 16-bit row offsets).
__global__ void __launch_bounds__(RT) k_rc_dict(int n, const int *__restrict__ ia, const int *__restrict__ ja, const double *__restrict__ a,
                                                unsigned char *__restrict__ codes, bool skip_stencil, unsigned char *__restrict__ tkind,
                                                PkHeader *__restrict__ thdr, unsigned *__restrict__ tbytes)
{
  __shared__ int                st[DS];   // 0 empty, 1 being written, 2 holds a key
  __shared__ int                sd[DS], sfirst[DS];
  __shared__ unsigned long long sb[DS];
  __shared__ unsigned char      scode[DS];
  __shared__ int                sia[TR + 1], list[RT];
  __shared__ int                ndist, ncomp, overflow, maxlen;
  const int t = blockIdx.x;
  if (skip_stencil && tkind[t] == 2) return;   // stencil tile (k_rc_stencil)
  const int r0 = t * TR, r1 = min(r0 + TR, n), nrows = r1 - r0;
  for (int s = threadIdx.x; s < DS; s += RT) {
    st[s]     = 0;
    sfirst[s] = INT_MAX;
  }
  for (int i = threadIdx.x; i <= nrows; i += RT) sia[i] = ia[r0 + i];
  if (threadIdx.x == 0) ndist = ncomp = overflow = maxlen = 0;
  __syncthreads();
  const int k0 = sia[0], k1 = sia[nrows], nnz = k1 - k0;
  volatile int                *vst = st, *vsd = sd, *vof = &overflow;
  volatile unsigned long long *vsb = sb;
  for (int k = k0 + threadIdx.x; k < k1 && !*vof; k += RT) {
    const int                d = ja[k] - (r0 + rc_row_of(sia, nrows, k));
    const unsigned long long b = dbits(a[k]);
    unsigned                 h = rc_hash(d, b);
    bool                     stop = false;
    for (;;) {
      const int s = vst[h];
      if (s == 0) {
        if (atomicCAS(&st[h], 0, 1) != 0) continue;
        vsd[h] = d;
        vsb[h] = b;
        __threadfence_block();
        atomicExch(&st[h], 2);
        atomicMin(&sfirst[h], k - k0);
        if (atomicAdd(&ndist, 1) >= 256) {
          *vof = 1;
          stop = true;
        }
        break;
      }
      if (s == 1) continue;   // another thread is writing this slot's key
      if (vsd[h] == d && vsb[h] == b) {
        atomicMin(&sfirst[h], k - k0);
        break;
      }
      h = (h + 1) & (DS - 1);
    }
    if (stop) break;
  }
  __syncthreads();
  if (overflow) {   // more than 256 distinct pairs: raw tile
    if (threadIdx.x == 0) {
      PkHeader H;
      H.kind    = 0;
      H.ndict   = 0;
      H.nnz     = (uint32_t)nnz;
      H.ulen    = 0xFFFF;
      H.nrows   = (uint16_t)nrows;
      H.pad     = 0;
      thdr[t]   = H;
      tkind[t]  = 0;
      tbytes[t] = (unsigned)pk_raw_bytes(nrows, nnz);
    }
    return;
  }
  for (int s = threadIdx.x; s < DS; s += RT)
    if (st[s] == 2) list[atomicAdd(&ncomp, 1)] = s;
  __syncthreads();
  const int nd = ndist;
  if (threadIdx.x < nd) {
    const int my = sfirst[list[threadIdx.x]];
    int       rank = 0;
    for (int j = 0; j < nd; j++) rank += (sfirst[list[j]] < my);
    scode[list[threadIdx.x]] = (unsigned char)rank;
  }
  __syncthreads();
  for (int k = k0 + threadIdx.x; k < k1; k += RT) {
    const int                d = ja[k] - (r0 + rc_row_of(sia, nrows, k));
    const unsigned long long b = dbits(a[k]);
    unsigned                 h = rc_hash(d, b);
    while (!(sd[h] == d && sb[h] == b && st[h] == 2)) h = (h + 1) & (DS - 1);
    codes[k] = scode[h];
  }
  const int len0 = sia[1] - sia[0];
  int       same = 1;
  if (threadIdx.x < nrows) {
    const int len = sia[threadIdx.x + 1] - sia[threadIdx.x];
    same          = (len == len0);
    atomicMax(&maxlen, len);
  }
  const bool uniform = __syncthreads_and(same);
  if (threadIdx.x == 0) {
    const bool uni    = uniform && len0 < 0xFFFF;
    const int  padded = nrows * maxlen;
    PkHeader   H;
    H.kind  = 1;
    H.nnz   = (uint32_t)nnz;
    H.nrows = (uint16_t)nrows;
    if (!uniform && maxlen <= 8 && nd <= 255 && padded <= nnz + nnz / 4 + 16) {
      H.ndict   = (uint16_t)(nd + 1);   // the skip code's (0, 0.0) slot
      H.ulen    = (uint16_t)maxlen;
      H.pad     = (uint32_t)nd + 1u;
      tbytes[t] = (unsigned)pk_coded_bytes(nd + 1, nrows, padded, true);
    } else {
      H.ndict   = (uint16_t)nd;
      H.ulen    = uni ? (uint16_t)len0 : (uint16_t)0xFFFF;
      H.pad     = 0;
      tbytes[t] = (unsigned)pk_coded_bytes(nd, nrows, nnz, uni);
    }
    thdr[t]  = H;
    tkind[t] = 1;
  }
}

// one tile of the blob (pack.cpp layout) into the zeroed blob
__global__ void __launch_bounds__(RT) k_rc_fill(int n, const int *__restrict__ ia, const int *__restrict__ ja, const double *__restrict__ a,
                                                const unsigned char *__restrict__ codes, const unsigned char *__restrict__ masks, const RcPat *__restrict__ tpat,
                                                const PkHeader *__restrict__ thdr, const unsigned *__restrict__ off, unsigned char *__restrict__ blob)
{
  __shared__ int sia[TR + 1];
  const int      t = blockIdx.x, r0 = t * TR, r1 = min(r0 + TR, n), nrows = r1 - r0;
  for (int i = threadIdx.x; i <= nrows; i += RT) sia[i] = ia[r0 + i];
  __syncthreads();
  const PkHeader H  = thdr[t];
  const int      k0 = sia[0], k1 = sia[nrows], nnz = k1 - k0;
  unsigned char *p  = blob + (size_t)off[t] * 16;
  if (threadIdx.x == 0) *(PkHeader *)p = H;
  if (H.kind == 2) {
    const int    L = H.ndict;
    const size_t o_val = sizeof(PkHeader), o_del = o_val + pk_up(L, 2) * 8, o_mask = o_del + pk_up(L, 4) * 4;
    if (threadIdx.x < L) {
      ((unsigned long long *)(p + o_val))[threadIdx.x] = tpat[t].b[threadIdx.x];
      ((int *)(p + o_del))[threadIdx.x]                = tpat[t].d[threadIdx.x];
    }
    if (threadIdx.x < nrows) p[o_mask + threadIdx.x] = masks[(size_t)r0 + threadIdx.x];
  } else if (H.kind == 1) {
    const int    nd = H.ndict, plen = H.pad ? H.ulen : 0, nd0 = plen ? nd - 1 : nd;
    const size_t o_val = sizeof(PkHeader), o_del = o_val + pk_up(nd, 2) * 8, o_ro = o_del + pk_up(nd, 4) * 4;
    const size_t o_code = o_ro + (H.ulen == 0xFFFF ? pk_up((size_t)nrows + 1, 8) * 2 : 0);
    double      *val = (double *)(p + o_val);
    int         *del = (int *)(p + o_del);
    // every entry stores its pair into its code's slot: the entries of one code carry the same pair, so the bytes do not depend on
    // which of them lands last
    for (int k = k0 + threadIdx.x; k < k1; k += RT) {
      const int c = codes[k];
      val[c]      = a[k];
      del[c]      = ja[k] - (r0 + rc_row_of(sia, nrows, k));
    }
    if (plen) {
      if (threadIdx.x < nrows) {
        unsigned char *rc  = p + o_code + (size_t)threadIdx.x * plen;
        const int      kr  = sia[threadIdx.x], len = sia[threadIdx.x + 1] - kr;
        for (int q = 0; q < plen; q++) rc[q] = q < len ? codes[kr + q] : (unsigned char)nd0;
      }
    } else {
      for (int k = k0 + threadIdx.x; k < k1; k += RT) p[o_code + (k - k0)] = codes[k];
    }
    if (H.ulen == 0xFFFF)
      for (int i = threadIdx.x; i <= nrows; i += RT) ((uint16_t *)(p + o_ro))[i] = (uint16_t)(sia[i] - k0);
  } else {
    size_t o = sizeof(PkHeader);
    for (int k = k0 + threadIdx.x; k < k1; k += RT) ((double *)(p + o))[k - k0] = a[k];
    o += pk_up(nnz, 2) * 8;
    for (int k = k0 + threadIdx.x; k < k1; k += RT) ((int *)(p + o))[k - k0] = ja[k];
    o += pk_up(nnz, 4) * 4;
    for (int i = threadIdx.x; i <= nrows; i += RT) ((uint16_t *)(p + o))[i] = (uint16_t)(sia[i] - k0);
  }
}

// ---- row split of a row-partitioned matrix ------------------------------------------------------------
__global__ void k_rc_split_count(int m, const int *__restrict__ ia, const int *__restrict__ ja, int c0, int c1, int *__restrict__ dcnt, int *__restrict__ ocnt)
{
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < m; r += gridDim.x * blockDim.x) {
    int nd = 0;
    for (int k = ia[r]; k < ia[r + 1]; k++) nd += (ja[k] >= c0 && ja[k] < c1);
    dcnt[r] = nd;
    ocnt[r] = ia[r + 1] - ia[r] - nd;
  }
}
__global__ void k_rc_split_fill(int m, const int *__restrict__ ia, const int *__restrict__ ja, const double *__restrict__ a, int c0, int c1,
                                const int *__restrict__ dia, const int *__restrict__ oia, int *__restrict__ dja, double *__restrict__ da,
                                int *__restrict__ orow, int *__restrict__ ogcol, double *__restrict__ oval)
{
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < m; r += gridDim.x * blockDim.x) {
    int pd = dia ? dia[r] : 0, po = oia[r];
    for (int k = ia[r]; k < ia[r + 1]; k++) {
      const int c = ja[k];
      if (c >= c0 && c < c1) {
        if (dja) {   // NULL: only the ghost entries are wanted
          dja[pd]  = c - c0;
          da[pd++] = a[k];
        }
      } else {
        orow[po]   = r;
        ogcol[po]  = c;
        oval[po++] = a[k];
      }
    }
  }
}

// exclusive prefix sum of m counts into out[0..m]: chunk sums, their prefix on the host, then each chunk scanned with its offset
constexpr int SC_PER = 16, SC_CHUNK = RT * SC_PER;
__global__ void __launch_bounds__(RT) k_rc_chunk_sum(int m, const int *__restrict__ cnt, long long *__restrict__ sums)
{
  __shared__ long long w[RT / 32];
  const int            base = blockIdx.x * SC_CHUNK;
  long long            s = 0;
  for (int i = threadIdx.x; i < SC_CHUNK && base + i < m; i += RT) s += cnt[base + i];
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) w[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    long long tot = 0;
    for (int q = 0; q < RT / 32; q++) tot += w[q];
    sums[blockIdx.x] = tot;
  }
}
__global__ void __launch_bounds__(RT) k_rc_chunk_scan(int m, const int *__restrict__ cnt, const long long *__restrict__ base_off, int *__restrict__ out)
{
  __shared__ long long ts[RT];
  const int            base = blockIdx.x * SC_CHUNK + threadIdx.x * SC_PER;
  int                  v[SC_PER];
  long long            s = 0;
  for (int q = 0; q < SC_PER; q++) {
    v[q] = (base + q < m) ? cnt[base + q] : 0;
    s += v[q];
  }
  ts[threadIdx.x] = s;
  __syncthreads();
  for (int o = 1; o < RT; o <<= 1) {   // inclusive scan of the thread sums
    const long long x = threadIdx.x >= o ? ts[threadIdx.x - o] : 0;
    __syncthreads();
    ts[threadIdx.x] += x;
    __syncthreads();
  }
  long long run = base_off[blockIdx.x] + ts[threadIdx.x] - s;
  if (blockIdx.x == 0 && threadIdx.x == 0) out[0] = 0;
  for (int q = 0; q < SC_PER && base + q < m; q++) {
    run += v[q];
    out[base + q + 1] = (int)run;
  }
}

int grid_for(int64_t work) { return (int)std::max<int64_t>(1, std::min<int64_t>((work + RT - 1) / RT, (int64_t)ctx().sm_count * 16)); }

template <class T>
struct DBuf {   // library scratch on the device, released at scope exit (stream-ordered)
  T *p = nullptr;
  ~DBuf() { dfree(p); }
  int alloc(size_t count) { return dmalloc(&p, std::max<size_t>(count, 1)); }
  T  *release()   // hand the buffer to its new owner
  {
    T *q = p;
    p    = nullptr;
    return q;
  }
};

int scan_counts(int m, const int *cnt, int *out, int64_t *total)
{
  cudaStream_t s = ctx().stream;
  const int    nch = std::max(1, (m + SC_CHUNK - 1) / SC_CHUNK);
  DBuf<long long> sums;
  PB_CHK(sums.alloc(nch));
  if (m > 0) {
    k_rc_chunk_sum<<<nch, RT, 0, s>>>(m, cnt, sums.p);
    PB_CUDA(cudaGetLastError());
  }
  std::vector<long long> h((size_t)nch, 0);
  PB_CUDA(cudaMemcpyAsync(h.data(), sums.p, sizeof(long long) * (size_t)nch, cudaMemcpyDeviceToHost, s));
  PB_CUDA(cudaStreamSynchronize(s));
  long long run = 0;
  for (int c = 0; c < nch; c++) {
    const long long x = h[c];
    h[c]              = run;
    run += (m > 0) ? x : 0;
  }
  if (run > INT_MAX) return err(PETSC_ERR_ARG_OUTOFRANGE, "device CSR: more than 2^31 - 1 non-zeros in one block");
  PB_CUDA(cudaMemcpyAsync(sums.p, h.data(), sizeof(long long) * (size_t)nch, cudaMemcpyHostToDevice, s));
  if (m > 0) {
    k_rc_chunk_scan<<<nch, RT, 0, s>>>(m, cnt, sums.p, out);
    PB_CUDA(cudaGetLastError());
  } else {
    PB_CUDA(cudaMemsetAsync(out, 0, sizeof(int), s));
  }
  PB_CUDA(cudaStreamSynchronize(s));   // h is a local
  *total = run;
  return 0;
}
}   // namespace

// the stencil pass over every tile (columns in [c0, c1)), then, when every tile passed and want_all, the all-stencil form: the patterns
// of the tiles where the pattern changes are deduped in tile order (pk_build / pk_stencil_windowed) and the pattern ids filled in.
// *all_done: C holds the all-stencil form.  Otherwise tkind / thdr / tbytes / tpat / masks describe the tiles for the blob.
struct TileScratch {
  DBuf<unsigned char> tkind, masks;   // masks: ntiles * 256 presence bytes and one zero tile (the stencil kernel's spare tile)
  DBuf<RcPat>         tpat;
  DBuf<PkHeader>      thdr;
  DBuf<unsigned>      tbytes, cnt;
  DBuf<unsigned long long> nwin_nnz;
};
static int stencil_pass(CsrDev &C, int n, const int *ia, const int *ja, const double *a, int c0, int c1, bool want_all, TileScratch &S, bool *all_done)
{
  *all_done = false;
  cudaStream_t s = ctx().stream;
  const int    ntiles = (n + TR - 1) / TR;
  PB_CHK(S.tpat.alloc(ntiles));
  PB_CHK(S.masks.alloc((size_t)ntiles * TR + TR));
  PB_CHK(S.nwin_nnz.alloc(1));
  PB_CUDA(cudaMemsetAsync(S.masks.p + (size_t)ntiles * TR, 0, TR, s));
  PB_CUDA(cudaMemsetAsync(S.cnt.p, 0, 2 * sizeof(unsigned), s));
  PB_CUDA(cudaMemsetAsync(S.nwin_nnz.p, 0, sizeof(unsigned long long), s));
  k_rc_stencil<<<ntiles, RT, 0, s>>>(n, ia, ja, a, c0, c1, S.masks.p, S.tpat.p, S.tkind.p, S.thdr.p, S.tbytes.p, S.cnt.p, S.nwin_nnz.p);
  PB_CUDA(cudaGetLastError());
  unsigned           nst = 0;
  unsigned long long nnz_win = 0;
  PB_CUDA(cudaMemcpyAsync(&nst, S.cnt.p, sizeof nst, cudaMemcpyDeviceToHost, s));
  PB_CUDA(cudaMemcpyAsync(&nnz_win, S.nwin_nnz.p, sizeof nnz_win, cudaMemcpyDeviceToHost, s));
  PB_CUDA(cudaStreamSynchronize(s));
  if (!want_all || nst != (unsigned)ntiles) return 0;
  DBuf<RcPat> rec;
  PB_CHK(rec.alloc(ntiles));
  k_rc_changes<<<grid_for(ntiles), RT, 0, s>>>(ntiles, S.tpat.p, rec.p, S.cnt.p + 1);
  PB_CUDA(cudaGetLastError());
  unsigned nrec = 0;
  PB_CUDA(cudaMemcpyAsync(&nrec, S.cnt.p + 1, sizeof nrec, cudaMemcpyDeviceToHost, s));
  PB_CUDA(cudaStreamSynchronize(s));
  std::vector<RcPat> h(nrec);
  PB_CUDA(cudaMemcpyAsync(h.data(), rec.p, sizeof(RcPat) * nrec, cudaMemcpyDeviceToHost, s));
  PB_CUDA(cudaStreamSynchronize(s));
  std::sort(h.begin(), h.end(), [](const RcPat &x, const RcPat &y) { return x.t < y.t; });
  std::vector<StPattern>     pats;
  std::vector<int>           run_t(nrec);
  std::vector<unsigned char> run_id(nrec);
  for (unsigned i = 0; i < nrec; i++) {
    const RcPat &T  = h[i];
    int          id = -1;
    for (int c = 0; c < (int)pats.size() && id < 0; c++) {
      const StPattern &Q = pats[(size_t)c];
      if (Q.L == T.L && !memcmp(Q.d, T.d, sizeof(int) * T.L) && !memcmp(Q.v, T.b, sizeof(double) * T.L)) id = c;
    }
    if (id < 0) {
      if ((int)pats.size() == PB_ST_MAXPAT) return 0;   // too many patterns
      StPattern P;
      memset(&P, 0, sizeof P);
      P.L = T.L;
      memcpy(P.d, T.d, sizeof(int) * T.L);
      memcpy(P.v, T.b, sizeof(double) * T.L);
      P.nwin = pattern_windows(P) + 1;
      id     = (int)pats.size();
      pats.push_back(P);
    }
    run_t[i]  = T.t;
    run_id[i] = (unsigned char)id;
  }
  int nwin = 0;
  for (const StPattern &P : pats) nwin = std::max(nwin, P.nwin);
  DBuf<int>           drt;
  DBuf<unsigned char> dri, dp;
  DBuf<StPattern>     dt;
  PB_CHK(drt.alloc(nrec));
  PB_CHK(dri.alloc(nrec));
  PB_CHK(dp.alloc((size_t)ntiles + 16));
  PB_CHK(dt.alloc(pats.size()));
  PB_CUDA(cudaMemcpyAsync(drt.p, run_t.data(), sizeof(int) * nrec, cudaMemcpyHostToDevice, s));
  PB_CUDA(cudaMemcpyAsync(dri.p, run_id.data(), nrec, cudaMemcpyHostToDevice, s));
  PB_CUDA(cudaMemcpyAsync(dt.p, pats.data(), sizeof(StPattern) * pats.size(), cudaMemcpyHostToDevice, s));
  PB_CUDA(cudaMemsetAsync(dp.p + ntiles, 0, 16, s));
  k_rc_fill_pid<<<grid_for(ntiles), RT, 0, s>>>(ntiles, (int)nrec, drt.p, dri.p, dp.p);
  PB_CUDA(cudaGetLastError());
  PB_CUDA(cudaStreamSynchronize(s));   // run_t / run_id / pats are locals
  C.nnz      = (int64_t)nnz_win;
  C.st_masks = S.masks.release();
  C.st_pid   = dp.release();
  C.st_pats  = dt.release();
  stencil_set_fields(C, pats, nwin, (size_t)ntiles * TR, (size_t)ntiles);
  *all_done = true;
  return 0;
}

static int scratch_alloc(TileScratch &S, int ntiles)
{
  PB_CHK(S.tkind.alloc(ntiles));
  PB_CHK(S.thdr.alloc(ntiles));
  PB_CHK(S.tbytes.alloc(ntiles));
  PB_CHK(S.cnt.alloc(2));
  return 0;
}

// the all-stencil form or packed tiles; *done = false when the matrix stays CSR (upload_csr's rules)
static int recode_packed(CsrDev &C, int n, int ncols, int cap, const int *ia, const int *ja, const double *a, bool *done)
{
  *done = false;
  if (cap > 65535) return 0;   // a tile's non-zeros do not fit the 16-bit row offsets: pk_build gives up
  cudaStream_t s = ctx().stream;
  const int    ntiles = (n + TR - 1) / TR;
  const char  *env_st = getenv("PERMON_B200_PACK_STENCIL"), *env_w = getenv("PERMON_B200_ST_WINDOWS");
  const bool   use_stencil = !(env_st && env_st[0] == '0');
  const bool   want_st = !(env_w && env_w[0] == '0') && n == ncols;
  TileScratch  S;
  PB_CHK(scratch_alloc(S, ntiles));
  if (use_stencil) {
    bool all = false;
    PB_CHK(stencil_pass(C, n, ia, ja, a, 0, INT_MAX, want_st, S, &all));
    if (all) {
      C.pk_coded = ntiles;
      *done      = true;
      return 0;
    }
  }
  // packed tiles
  DBuf<unsigned char> codes;
  PB_CHK(codes.alloc((size_t)C.nnz));
  k_rc_dict<<<ntiles, RT, 0, s>>>(n, ia, ja, a, codes.p, use_stencil, S.tkind.p, S.thdr.p, S.tbytes.p);
  PB_CUDA(cudaGetLastError());
  std::vector<unsigned>      hb((size_t)ntiles);
  std::vector<unsigned char> hk((size_t)ntiles);
  PB_CUDA(cudaMemcpyAsync(hb.data(), S.tbytes.p, sizeof(unsigned) * (size_t)ntiles, cudaMemcpyDeviceToHost, s));
  PB_CUDA(cudaMemcpyAsync(hk.data(), S.tkind.p, (size_t)ntiles, cudaMemcpyDeviceToHost, s));
  PB_CUDA(cudaStreamSynchronize(s));
  std::vector<unsigned> off((size_t)ntiles + 1);
  size_t                tot = 0;
  int                   max_tile = 0;
  int64_t               ncoded = 0;
  for (int t = 0; t < ntiles; t++) {
    off[t] = (unsigned)(tot / 16);
    tot += hb[t];
    max_tile = std::max(max_tile, (int)hb[t]);
    ncoded += (hk[t] != 0);
  }
  if (tot / 16 > 0xFFFFFFFFull || (!getenv("PERMON_B200_KEEP_RAW_TILES") && ncoded * 3 < ntiles)) return 0;   // CSR (see upload_csr)
  off[ntiles] = (unsigned)(tot / 16);
  DBuf<unsigned char> dblob;
  DBuf<unsigned>      doff;
  PB_CHK(dblob.alloc(tot + 16));
  PB_CHK(doff.alloc(off.size()));
  PB_CUDA(cudaMemsetAsync(dblob.p, 0, tot + 16, s));   // padding bytes are defined
  PB_CUDA(cudaMemcpyAsync(doff.p, off.data(), sizeof(unsigned) * off.size(), cudaMemcpyHostToDevice, s));
  k_rc_fill<<<ntiles, RT, 0, s>>>(n, ia, ja, a, codes.p, S.masks.p, S.tpat.p, S.thdr.p, doff.p, dblob.p);
  PB_CUDA(cudaGetLastError());
  PB_CUDA(cudaStreamSynchronize(s));   // off is a local
  C.pk       = dblob.release();
  C.pk_off   = doff.release();
  C.pk_max   = max_tile;
  C.pk_bytes = (int64_t)off.back() * 16 + (int64_t)sizeof(unsigned) * (int64_t)off.size();
  C.pk_coded = ncoded;
  C.kind     = 3;
  const char *stg = getenv("PERMON_B200_STAGES");
  C.stages        = stg ? atoi(stg) : 3;
  *done           = true;
  return 0;
}

int recode_csr_dev(CsrDev &C, int nrows, int ncols, const int *d_ia, const int *d_ja, const double *d_a, int **own_ia, int **own_ja, double **own_a)
{
  cudaStream_t s = ctx().stream;
  int          nnz32 = 0, stats[2] = {0, 0};
  DBuf<int>    dstats;
  PB_CHK(dstats.alloc(2));
  PB_CUDA(cudaMemsetAsync(dstats.p, 0, 2 * sizeof(int), s));
  if (nrows > 0) {
    k_rc_stats<<<grid_for(nrows), RT, 0, s>>>(nrows, d_ia, dstats.p);
    PB_CUDA(cudaGetLastError());
  }
  PB_CUDA(cudaMemcpyAsync(&nnz32, d_ia + nrows, sizeof(int), cudaMemcpyDeviceToHost, s));
  PB_CUDA(cudaMemcpyAsync(stats, dstats.p, sizeof stats, cudaMemcpyDeviceToHost, s));
  PB_CUDA(cudaStreamSynchronize(s));
  const int64_t nnz = nnz32;
  C.n     = nrows;
  C.ncols = ncols;
  C.nnz   = nnz;
  spmv_decide(C, stats[0], stats[1]);
  if (C.kind == 2 && nrows >= 64 && !getenv("PERMON_B200_SPMV")) {
    bool done = false;
    PB_CHK(recode_packed(C, nrows, ncols, stats[1], d_ia, d_ja, d_a, &done));
    if (done) return 0;
  }
  C.nnz_alloc = nnz + 8;
  C.ia_alloc  = nrows + 1 + 8;
  if (own_ia && own_ja && own_a) {
    // library-owned arrays with the padding below already in place: adopted as they are
    C.ia    = *own_ia;
    C.ja    = *own_ja;
    C.a     = *own_a;
    *own_ia = *own_ja = nullptr;
    *own_a  = nullptr;
  } else {
    DBuf<int>    dia, dja;
    DBuf<double> da;
    // 8 elements of padding: the TMA kernel copies 16-byte aligned, 16-byte granular tile ranges
    PB_CHK(dia.alloc((size_t)(nrows + 1 + 8)));
    PB_CHK(dja.alloc((size_t)(nnz + 8)));
    PB_CHK(da.alloc((size_t)(nnz + 8)));
    PB_CUDA(cudaMemsetAsync(dia.p + nrows + 1, 0, sizeof(int) * 8, s));
    PB_CUDA(cudaMemsetAsync(dja.p + nnz, 0, sizeof(int) * 8, s));
    PB_CUDA(cudaMemsetAsync(da.p + nnz, 0, sizeof(double) * 8, s));
    PB_CUDA(cudaMemcpyAsync(dia.p, d_ia, sizeof(int) * (size_t)(nrows + 1), cudaMemcpyDeviceToDevice, s));
    PB_CUDA(cudaMemcpyAsync(dja.p, d_ja, sizeof(int) * (size_t)nnz, cudaMemcpyDeviceToDevice, s));
    PB_CUDA(cudaMemcpyAsync(da.p, d_a, sizeof(double) * (size_t)nnz, cudaMemcpyDeviceToDevice, s));
    C.ia = dia.release();
    C.ja = dja.release();
    C.a  = da.release();
  }
  if (C.kind == 1 && nnz >= (1 << 20) && !getenv("PERMON_B200_SPMV") && !getenv("PERMON_B200_NOELL")) {
    const int        ntiles = (nrows + TR - 1) / TR;
    DBuf<int>        dlt;
    std::vector<int> lt((size_t)ntiles);
    PB_CHK(dlt.alloc(ntiles));
    k_rc_tile_maxrow<<<ntiles, RT, 0, s>>>(nrows, C.ia, dlt.p);
    PB_CUDA(cudaGetLastError());
    PB_CUDA(cudaMemcpyAsync(lt.data(), dlt.p, sizeof(int) * (size_t)ntiles, cudaMemcpyDeviceToHost, s));
    PB_CUDA(cudaStreamSynchronize(s));
    PB_CHK(csr_to_tile_ell_widths(C, lt));
  }
  return 0;
}

int recode_stencil_window_dev(CsrDev &C, int m, const int *d_ia, const int *d_ja, const double *d_a, int c0, int ncols, bool *done)
{
  *done = false;
  if (m <= 0) return 0;
  TileScratch S;
  PB_CHK(scratch_alloc(S, (m + TR - 1) / TR));
  C.n     = m;
  C.ncols = ncols;
  PB_CHK(stencil_pass(C, m, d_ia, d_ja, d_a, c0, c0 + ncols, true, S, done));
  if (*done) C.pk_coded = (m + TR - 1) / TR;
  return 0;
}

int split_rows_dev(int m, const int *d_ia, const int *d_ja, const double *d_a, int c0, int ncols, bool want_diag, int **dia_out, int **dja_out,
                   double **da_out, OffDiagEntries &off)
{
  cudaStream_t s = ctx().stream;
  DBuf<int>    dcnt, ocnt, oia, orow, ogcol, dia, dja;
  DBuf<double> oval, da;
  PB_CHK(dcnt.alloc(m));
  PB_CHK(ocnt.alloc(m));
  PB_CHK(oia.alloc((size_t)m + 1));
  if (m > 0) {
    k_rc_split_count<<<grid_for(m), RT, 0, s>>>(m, d_ia, d_ja, c0, c0 + ncols, dcnt.p, ocnt.p);
    PB_CUDA(cudaGetLastError());
  }
  int64_t nd = 0, no = 0;
  if (want_diag) {   // with the padding recode_csr_dev expects of arrays it adopts
    PB_CHK(dia.alloc((size_t)m + 1 + 8));
    PB_CHK(scan_counts(m, dcnt.p, dia.p, &nd));
    PB_CHK(dja.alloc((size_t)nd + 8));
    PB_CHK(da.alloc((size_t)nd + 8));
    PB_CUDA(cudaMemsetAsync(dia.p + m + 1, 0, sizeof(int) * 8, s));
    PB_CUDA(cudaMemsetAsync(dja.p + nd, 0, sizeof(int) * 8, s));
    PB_CUDA(cudaMemsetAsync(da.p + nd, 0, sizeof(double) * 8, s));
  }
  PB_CHK(scan_counts(m, ocnt.p, oia.p, &no));
  PB_CHK(orow.alloc((size_t)no));
  PB_CHK(ogcol.alloc((size_t)no));
  PB_CHK(oval.alloc((size_t)no));
  if (m > 0) {
    k_rc_split_fill<<<grid_for(m), RT, 0, s>>>(m, d_ia, d_ja, d_a, c0, c0 + ncols, dia.p, oia.p, dja.p, da.p, orow.p, ogcol.p, oval.p);
    PB_CUDA(cudaGetLastError());
  }
  off.row.resize((size_t)no);
  off.gcol.resize((size_t)no);
  off.val.resize((size_t)no);
  PB_CUDA(cudaMemcpyAsync(off.row.data(), orow.p, sizeof(int) * (size_t)no, cudaMemcpyDeviceToHost, s));
  PB_CUDA(cudaMemcpyAsync(off.gcol.data(), ogcol.p, sizeof(int) * (size_t)no, cudaMemcpyDeviceToHost, s));
  PB_CUDA(cudaMemcpyAsync(off.val.data(), oval.p, sizeof(double) * (size_t)no, cudaMemcpyDeviceToHost, s));
  PB_CUDA(cudaStreamSynchronize(s));
  if (want_diag) {
    *dia_out = dia.release();
    *dja_out = dja.release();
    *da_out  = da.release();
  }
  return 0;
}

}   // namespace pb
