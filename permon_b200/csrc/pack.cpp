// Packed tile format of a CSR matrix ("dictionary-coded CSR tiles"), built once on the host at upload time.
//
// The MPGP iteration is HBM-bound and after fusion the matrix stream is the largest operand of K_A / K_A'
// (12 bytes per non-zero in CSR).  PDE Hessians repeat a small set of (column offset, value) pairs over and
// over -- 5 pairs for the whole 5-point Laplacian, a few dozen for a two-material finite-volume operator.  Each
// 256-row tile therefore carries its own dictionary of distinct (col - row, value) pairs and one byte per
// non-zero that indexes it; the kernel rebuilds col = row + delta and multiplies by the dictionary value, in
// storage order, so the row sums are bit-identical to the CSR kernels'.  A tile with more than 256 distinct pairs
// is stored raw (values + absolute columns) in the same blob, so one kernel handles any matrix.
//
// Tile blob (16-byte aligned, fetched with ONE bulk copy):
//   PkHeader (16 B)
//   coded: double val[nd2]            nd2 = ndict rounded up to 2
//          int    delta[nd4]          nd4 = ndict rounded up to 4
//          u16    rowoff[ro8]         only when the rows differ in length (ulen == 0xFFFF); ro8 = nrows+1 up to 8
//          u8     code[nnz16]         nnz rounded up to 16
//   Short ragged rows (longest <= 8, e.g. stencil rows next to a grid boundary) are padded to a common length with a
//   "skip" code (= ndict, stored in the header as pad = code + 1; its dictionary slot is (0, 0.0) and is never multiplied),
//   so that the kernel's unrolled equal-length path handles them too.
//   raw:   double a[nnz2] ; int ja[nnz4] ; u16 rowoff[ro8]
//   stencil (kind 2): double val[L2] ; int delta[L4] ; u8 present[nrows16]
//          every row of the tile is the tile's PATTERN -- the L <= 8 (col - row, value) pairs of its longest row, in storage order --
//          with some entries missing (constant-coefficient stencils: rows next to a grid boundary lack the neighbours that fall
//          outside); one presence byte per ROW replaces the code byte per non-zero, and the kernel reads deltas and values as
//          warp-uniform operands.  PERMON_B200_PACK_STENCIL=0 turns the form off (A/B measurements, tests of the coded form).
#include "device.h"
#include <omp.h>
#include <algorithm>
#include <cstring>
#include <vector>

namespace pb {

static inline size_t up(size_t v, size_t a) { return pk_up(v, a); }

// windows of a pattern: consecutive deltas within PB_ST_SPAN of the window's first delta share one; returns the last window index
int pattern_windows(StPattern &P)
{
  int w = -1, first = 0;
  for (int j = 0; j < P.L; j++) {
    if (w < 0 || P.d[j] - first > PB_ST_SPAN) {
      w++;
      first    = P.d[j];
      P.wlo[w] = (first & 1) ? first - 1 : first;   // even: 16-byte aligned copies (floor for negative odd values too)
    }
    int hi = P.d[j] + TR;
    if (hi & 1) hi++;
    P.wlen[w] = hi - P.wlo[w];
    P.erel[j] = w * PB_ST_WCAP + (P.d[j] - P.wlo[w]) * 8;
  }
  return w;
}
namespace {
struct TileDict {
  // open addressing over (delta, value bits); 1024 slots for at most 256 entries
  static constexpr int SLOTS = 1024;
  int                  slot_code[SLOTS];
  int                  delta[256];
  uint64_t             bits[256];
  int                  n;
  void reset()
  {
    n = 0;
    for (int s = 0; s < SLOTS; s++) slot_code[s] = -1;
  }
  // returns the code, or -1 when the dictionary is full
  int lookup(int d, uint64_t b)
  {
    uint64_t h = (b ^ (b >> 29)) * 0x9E3779B97F4A7C15ull + (uint64_t)(uint32_t)d * 0xC2B2AE3D27D4EB4Full;
    int      s = (int)((h >> 40) & (SLOTS - 1));
    for (;;) {
      const int c = slot_code[s];
      if (c < 0) {
        if (n == 256) return -1;
        slot_code[s] = n;
        delta[n]     = d;
        bits[n]      = b;
        return n++;
      }
      if (delta[c] == d && bits[c] == b) return c;
      s = (s + 1) & (SLOTS - 1);
    }
  }
};
}   // namespace

// row `c` (columns jc, values ac, len entries) has the same (column - row, value) list as the row before it (jp, ap): every column is the
// previous row's + 1 and the value bits agree.  A previous row that passed the stencil scan is sorted, so this one is sorted as well.
static inline bool row_is_shift_of(const int *jc, const double *ac, const int *jp, const double *ap, int len)
{
  if (len <= 0) return false;
  uint64_t acc = 0;   // branch-free: OR of the value-bit differences and of (column - previous column - 1)
  for (int k = 0; k < len; k++) {
    uint64_t x, y;
    memcpy(&x, ac + k, 8);
    memcpy(&y, ap + k, 8);
    acc |= (x ^ y) | (uint64_t)(uint32_t)(jc[k] - jp[k] - 1);
  }
  return acc == 0;
}

// h_off: ntiles+1 offsets in units of 16 bytes.  Returns 0 on success; `packed` false when packing is not applicable
// (a tile whose non-zero count or row lengths do not fit the 16-bit row offsets).
//
// Pass 1 (parallel over tiles) classifies every tile, builds its dictionary and writes the code bytes into a scratch array; the
// k-th entry of a row is first compared with the k-th entry of the previous row (a hit for almost every entry of a stencil
// matrix), the hash table is only consulted on a miss.  Pass 2 lays the blobs out: dictionary, row offsets and code bytes are
// copied, nothing is hashed again.
// st (optional): when every tile is a stencil tile and the matrix has at most PB_ST_MAXPAT patterns, the all-stencil form (device.h)
// is returned there; with want_blob == false the tile blobs are then not built at all.
int pk_build(int n, const int *ia, const int *ja, const double *a, RawBuf &blob, std::vector<unsigned> &h_off, int &max_tile_bytes,
             int64_t &ncoded, bool &packed, StencilHost *st, bool want_blob)
{
  if (st) st->valid = false;
  const int ntiles = (n + TR - 1) / TR;
  packed           = false;
  h_off.assign((size_t)ntiles + 1, 0);
  std::vector<unsigned>      tbytes(ntiles, 0);
  std::vector<unsigned char> tkind(ntiles, 0);
  std::vector<uint16_t>      tnd(ntiles, 0);
  std::vector<unsigned char> tpad(ntiles, 0);    // common (padded) row length of ragged short-row tiles, 0 = no padding
  std::vector<unsigned char> tuni(ntiles, 0);    // all rows of the tile have the same length
  std::vector<int>           tthr(ntiles, 0);    // which thread's arena holds the tile's dictionary ...
  std::vector<size_t>        tdoff(ntiles, 0);   // ... and where
  const int64_t  nnz_all = n > 0 ? ia[n] : 0;
  unsigned char *codes_tmp = (unsigned char *)malloc((size_t)std::max<int64_t>(nnz_all, 1) + (size_t)std::max(n, 1));
  if (!codes_tmp) return 55;
  unsigned char *masks_tmp = codes_tmp + (size_t)std::max<int64_t>(nnz_all, 1);   // one presence byte per row (stencil tiles)
  const char    *env_st = getenv("PERMON_B200_PACK_STENCIL");
  const bool     use_stencil = !(env_st && env_st[0] == '0');
  const int nthr = omp_get_max_threads();
  std::vector<std::vector<int>>      arena_d(nthr);
  std::vector<std::vector<uint64_t>> arena_b(nthr);
  bool    bad = false;
  int64_t coded = 0;
#pragma omp parallel reduction(|| : bad) reduction(+ : coded)
  {
    TileDict               D;
    const int              me = omp_get_thread_num();
    std::vector<int>      &ad = arena_d[me];
    std::vector<uint64_t> &ab = arena_b[me];
#pragma omp for schedule(dynamic, 64)
    for (int t = 0; t < ntiles; t++) {
      const int r0 = t * TR, r1 = std::min(r0 + TR, n);
      const int k0 = ia[r0], k1 = ia[r1], nnz = k1 - k0;
      if (nnz > 65535) {
        bad = true;
        continue;
      }
      if (use_stencil) {
        // stencil form: the pattern is the ordered union of the rows' (delta, value) pairs -- rows must be sorted by column, a delta
        // must always carry the same value bits, and the union must not exceed 8 entries; every row is then a sub-sequence of it
        int      L = 0, pd[8];
        uint64_t pb[8];
        bool     st = (nnz > 0);
        // a row whose columns are the previous row's + 1 with the same value bits has the previous row's (delta, value) list: nothing to
        // merge and the same presence byte (almost every row of a grid operator: the scan then costs two compares per non-zero)
        unsigned char same[TR];
        int           prev_k = 0, prev_len = -1;
        for (int r = r0; r < r1 && st; r++) {
          const int rk = ia[r], rlen = ia[r + 1] - rk;
          same[r - r0] = (rlen == prev_len) && row_is_shift_of(ja + rk, a + rk, ja + prev_k, a + prev_k, rlen);
          prev_k       = rk;
          prev_len     = rlen > 0 ? rlen : -1;
          if (same[r - r0]) continue;
          int j = 0, prev_d = 0;
          for (int k = ia[r]; k < ia[r + 1]; k++) {
            uint64_t b;
            memcpy(&b, &a[k], 8);
            const int d = ja[k] - r;
            if (k > ia[r] && d <= prev_d) {
              st = false;
              break;
            }
            prev_d = d;
            while (j < L && pd[j] < d) j++;
            if (j < L && pd[j] == d) {
              if (pb[j] != b) {
                st = false;
                break;
              }
            } else {
              if (L == 8) {
                st = false;
                break;
              }
              for (int q = L; q > j; q--) {
                pd[q] = pd[q - 1];
                pb[q] = pb[q - 1];
              }
              pd[j] = d;
              pb[j] = b;
              L++;
            }
            j++;
          }
        }
        if (st) {
          for (int r = r0; r < r1; r++) {
            if (same[r - r0]) {
              masks_tmp[r] = masks_tmp[r - 1];
              continue;
            }
            int      j = 0;
            unsigned m = 0;
            for (int k = ia[r]; k < ia[r + 1]; k++) {
              const int d = ja[k] - r;
              while (pd[j] != d) j++;
              m |= 1u << j;
              j++;
            }
            masks_tmp[r] = (unsigned char)m;
          }
          tkind[t] = 2;
          tnd[t]   = (uint16_t)L;
          tthr[t]  = me;
          tdoff[t] = ad.size();
          ad.insert(ad.end(), pd, pd + L);
          ab.insert(ab.end(), pb, pb + L);
          tbytes[t] = (unsigned)pk_stencil_bytes(L, r1 - r0);
          coded++;
          continue;
        }
      }
      D.reset();
      bool      ok = true, uniform = true;
      const int len0 = ia[r0 + 1] - ia[r0];
      int       maxlen = 0, prev_len = 0;
      const unsigned char *prev = nullptr;
      for (int r = r0; r < r1 && ok; r++) {
        const int      len = ia[r + 1] - ia[r];
        unsigned char *rc = codes_tmp + ia[r];
        if (len != len0) uniform = false;
        if (len > maxlen) maxlen = len;
        for (int k = 0; k < len; k++) {
          uint64_t b;
          memcpy(&b, &a[ia[r] + k], 8);
          const int d = ja[ia[r] + k] - r;
          if (k < prev_len && D.delta[prev[k]] == d && D.bits[prev[k]] == b) {
            rc[k] = prev[k];
            continue;
          }
          const int c = D.lookup(d, b);
          if (c < 0) {
            ok = false;
            break;
          }
          rc[k] = (unsigned char)c;
        }
        prev     = rc;
        prev_len = len;
      }
      if (ok) {
        tkind[t] = 1;
        tnd[t]   = (uint16_t)D.n;
        tuni[t]  = uniform && len0 < 0xFFFF;
        tthr[t]  = me;
        tdoff[t] = ad.size();
        ad.insert(ad.end(), D.delta, D.delta + D.n);
        ab.insert(ab.end(), D.bits, D.bits + D.n);
        const int padded = (r1 - r0) * maxlen;
        if (!uniform && maxlen <= 8 && D.n <= 255 && padded <= nnz + nnz / 4 + 16) {
          tpad[t]   = (unsigned char)maxlen;
          tbytes[t] = (unsigned)pk_coded_bytes(D.n + 1, r1 - r0, padded, true);
        } else {
          tbytes[t] = (unsigned)pk_coded_bytes(D.n, r1 - r0, nnz, tuni[t]);
        }
        coded++;
      } else {
        tkind[t]  = 0;
        tbytes[t] = (unsigned)pk_raw_bytes(r1 - r0, nnz);
      }
    }
  }
  if (bad) {
    free(codes_tmp);
    return 0;
  }
  if (st && ntiles > 0) {
    // all-stencil form: dedupe the tiles' patterns (a handful for a structured grid), then lay out the windows of each
    bool all = true;
    for (int t = 0; t < ntiles && all; t++) all = (tkind[t] == 2);
    if (all) {
      st->pats.clear();
      st->pid.assign((size_t)ntiles, 0);
      for (int t = 0; t < ntiles && all; t++) {
        const int       L = tnd[t];
        const int      *pd = arena_d[tthr[t]].data() + tdoff[t];
        const uint64_t *pb = arena_b[tthr[t]].data() + tdoff[t];
        int             id = -1;
        // the previous tile's pattern first: consecutive tiles almost always share it
        const int prev = t > 0 ? st->pid[(size_t)t - 1] : 0;
        for (int c = 0; c < (int)st->pats.size() && id < 0; c++) {
          const int        q = (c == 0) ? prev : (c <= prev ? c - 1 : c);
          if (q >= (int)st->pats.size()) continue;
          const StPattern &P = st->pats[q];
          if (P.L == L && !memcmp(P.d, pd, sizeof(int) * L) && !memcmp(P.v, pb, sizeof(double) * L)) id = q;
        }
        if (id < 0) {
          if ((int)st->pats.size() == PB_ST_MAXPAT) {
            all = false;
            break;
          }
          StPattern P;
          memset(&P, 0, sizeof P);
          P.L = L;
          memcpy(P.d, pd, sizeof(int) * L);
          memcpy(P.v, pb, sizeof(double) * L);
          int w = pattern_windows(P);
          P.nwin = w + 1;
          id     = (int)st->pats.size();
          st->pats.push_back(P);
        }
        st->pid[(size_t)t] = (unsigned char)id;
      }
      if (all && st->masks.alloc((size_t)ntiles * TR)) {
        memcpy(st->masks.data(), masks_tmp, (size_t)n);
        memset(st->masks.data() + n, 0, (size_t)ntiles * TR - (size_t)n);
        st->nwin = 0;
        for (const StPattern &P : st->pats) st->nwin = std::max(st->nwin, P.nwin);
        st->valid = true;
        if (!want_blob) {
          free(codes_tmp);
          ncoded = coded;
          packed = true;
          return 0;
        }
      }
    }
  }
  size_t tot = 0;
  max_tile_bytes = 0;
  for (int t = 0; t < ntiles; t++) {
    h_off[t] = (unsigned)(tot / 16);
    tot += tbytes[t];
    if ((int)tbytes[t] > max_tile_bytes) max_tile_bytes = (int)tbytes[t];
  }
  if (tot / 16 > 0xFFFFFFFFull) {
    free(codes_tmp);
    return 0;
  }
  h_off[ntiles] = (unsigned)(tot / 16);
  if (!blob.alloc(tot + 16)) {
    free(codes_tmp);
    return 55;
  }
  memset(blob.data() + tot, 0, 16);
#pragma omp parallel for schedule(dynamic, 64)
  for (int t = 0; t < ntiles; t++) {
    const int      r0 = t * TR, r1 = std::min(r0 + TR, n), nrows = r1 - r0;
    const int      k0 = ia[r0], k1 = ia[r1], nnz = k1 - k0;
    unsigned char *p = blob.data() + (size_t)h_off[t] * 16;
    memset(p, 0, tbytes[t]);   // padding bytes are defined
    PkHeader H;
    memset(&H, 0, sizeof H);
    H.kind  = tkind[t];
    H.nnz   = (uint32_t)nnz;
    H.nrows = (uint16_t)nrows;
    if (tkind[t] == 2) {
      const int L = tnd[t];
      H.ndict = (uint16_t)L;
      H.ulen  = (uint16_t)L;
      const size_t o_val = sizeof(PkHeader), o_del = o_val + up(L, 2) * 8, o_mask = o_del + up(L, 4) * 4;
      memcpy(p + o_val, arena_b[tthr[t]].data() + tdoff[t], (size_t)L * 8);
      memcpy(p + o_del, arena_d[tthr[t]].data() + tdoff[t], (size_t)L * 4);
      memcpy(p + o_mask, masks_tmp + r0, (size_t)nrows);
    } else if (tkind[t] == 1) {
      const int plen = tpad[t];                     // > 0: rows padded to this length with the skip code
      const int nd0 = tnd[t], nd = nd0 + (plen ? 1 : 0);   // the skip code owns a (0, 0.0) slot at the end of the dictionary
      H.ndict = (uint16_t)nd;
      H.ulen  = plen ? (uint16_t)plen : (tuni[t] ? (uint16_t)(ia[r0 + 1] - ia[r0]) : (uint16_t)0xFFFF);
      H.pad   = plen ? (uint32_t)nd0 + 1u : 0u;
      const size_t o_val = sizeof(PkHeader), o_del = o_val + up(nd, 2) * 8, o_ro = o_del + up(nd, 4) * 4;
      const size_t o_code = o_ro + (H.ulen == 0xFFFF ? up((size_t)nrows + 1, 8) * 2 : 0);
      unsigned char *codes = p + o_code;
      memcpy(p + o_val, arena_b[tthr[t]].data() + tdoff[t], (size_t)nd0 * 8);
      memcpy(p + o_del, arena_d[tthr[t]].data() + tdoff[t], (size_t)nd0 * 4);
      if (plen) {
        for (int r = r0; r < r1; r++) {
          unsigned char *rc = codes + (size_t)(r - r0) * plen;
          const int      len = ia[r + 1] - ia[r];
          memcpy(rc, codes_tmp + ia[r], (size_t)len);
          for (int k = len; k < plen; k++) rc[k] = (unsigned char)nd0;
        }
      } else if (nnz) {
        memcpy(codes, codes_tmp + k0, (size_t)nnz);
      }
      if (H.ulen == 0xFFFF) {
        uint16_t *ro = (uint16_t *)(p + o_ro);
        for (int r = r0; r <= r1; r++) ro[r - r0] = (uint16_t)(ia[r] - k0);
      }
    } else {
      H.ndict = 0;
      H.ulen  = 0xFFFF;
      size_t o = sizeof(PkHeader);
      if (nnz) memcpy(p + o, a + k0, (size_t)nnz * 8);
      o += up(nnz, 2) * 8;
      if (nnz) memcpy(p + o, ja + k0, (size_t)nnz * 4);
      o += up(nnz, 4) * 4;
      uint16_t *ro = (uint16_t *)(p + o);
      for (int r = r0; r <= r1; r++) ro[r - r0] = (uint16_t)(ia[r] - k0);
    }
    memcpy(p, &H, sizeof H);
  }
  free(codes_tmp);
  ncoded = coded;
  packed = true;
  return 0;
}

// All-stencil form of the DIAGONAL BLOCK of a row-partitioned matrix, straight from the caller's CSR with GLOBAL column indices: an
// entry belongs to the block when coff <= col < coff + ncols (its local column is col - coff), every other entry is a ghost entry and
// is appended to `off` (row, global column, value; storage order kept per row).  One pass over the arrays -- no intermediate copy of the
// diagonal block is made.  Returns with st.valid == false when some tile is not a stencil tile or there are too many patterns (the
// caller then splits the matrix the general way).  nnz_diag: entries of the block.
int pk_stencil_windowed(int n, const int *ia, const int *ja, const double *a, int coff, int ncols, StencilHost &st, OffDiagEntries &off, int64_t &nnz_diag)
{
  const int ntiles = (n + TR - 1) / TR;
  st.valid  = false;
  nnz_diag  = 0;
  off.row.clear();
  off.gcol.clear();
  off.val.clear();
  if (ntiles == 0) return 0;
  if (!st.masks.alloc((size_t)ntiles * TR)) return 55;
  std::vector<StPattern> tpat((size_t)ntiles);
  const int nthr = omp_get_max_threads();
  std::vector<OffDiagEntries> toff((size_t)nthr);
  bool    ok = true;
  int64_t nd = 0;
#pragma omp parallel reduction(&& : ok) reduction(+ : nd)
  {
    OffDiagEntries &mine = toff[(size_t)omp_get_thread_num()];
#pragma omp for schedule(static)
    for (int t = 0; t < ntiles; t++) {
      if (!ok) continue;
      const int r0 = t * TR, r1 = std::min(r0 + TR, n);
      int       L = 0, pd[8];
      uint64_t  pb[8];
      bool      st_ok = true;
      unsigned char *mk = st.masks.data() + (size_t)t * TR;
      unsigned char  same[TR];   // same (delta, value) list as the previous row (see pk_build)
      int            prev_k = 0, prev_len = -1;
      for (int r = r0; r < r1 && st_ok; r++) {
        const int rk = ia[r], rlen = ia[r + 1] - rk;
        // only rows without ghost columns qualify: the previous row had none (prev_len is reset otherwise) and this row's first / last
        // column (sorted: checked for the previous row, whose shift this one is) lie inside the diagonal block
        same[r - r0] = (rlen == prev_len) && ja[rk] - coff >= 0 && ja[rk + rlen - 1] - coff < ncols && row_is_shift_of(ja + rk, a + rk, ja + prev_k, a + prev_k, rlen);
        prev_k       = rk;
        prev_len     = rlen > 0 ? rlen : -1;
        if (same[r - r0]) {
          nd += rlen;
          continue;
        }
        int  j = 0, prev_d = 0;
        bool first = true;
        for (int k = ia[r]; k < ia[r + 1]; k++) {
          const int c = ja[k] - coff;
          if (c < 0 || c >= ncols) {   // ghost column
            mine.row.push_back(r);
            mine.gcol.push_back(ja[k]);
            mine.val.push_back(a[k]);
            prev_len = -1;             // the next row is scanned entry by entry
            continue;
          }
          uint64_t b;
          memcpy(&b, &a[k], 8);
          const int d = c - r;
          if (!first && d <= prev_d) {
            st_ok = false;
            break;
          }
          first  = false;
          prev_d = d;
          while (j < L && pd[j] < d) j++;
          if (j < L && pd[j] == d) {
            if (pb[j] != b) {
              st_ok = false;
              break;
            }
          } else {
            if (L == 8) {
              st_ok = false;
              break;
            }
            for (int q = L; q > j; q--) {
              pd[q] = pd[q - 1];
              pb[q] = pb[q - 1];
            }
            pd[j] = d;
            pb[j] = b;
            L++;
          }
          j++;
          nd++;
        }
      }
      if (!st_ok || L == 0) {
        ok = false;
        continue;
      }
      for (int r = r0; r < r1; r++) {   // presence bytes against the final pattern of the tile
        if (same[r - r0]) {
          mk[r - r0] = mk[r - r0 - 1];
          continue;
        }
        int      j = 0;
        unsigned m = 0;
        for (int k = ia[r]; k < ia[r + 1]; k++) {
          const int c = ja[k] - coff;
          if (c < 0 || c >= ncols) continue;
          const int d = c - r;
          while (pd[j] != d) j++;
          m |= 1u << j;
          j++;
        }
        mk[r - r0] = (unsigned char)m;
      }
      for (int r = r1; r < r0 + TR; r++) mk[r - r0] = 0;
      StPattern &P = tpat[(size_t)t];
      memset(&P, 0, sizeof P);
      P.L = L;
      memcpy(P.d, pd, sizeof(int) * L);
      memcpy(P.v, pb, sizeof(double) * L);
    }
  }
  if (!ok) return 0;
  // dedupe the tiles' patterns
  st.pats.clear();
  st.pid.assign((size_t)ntiles, 0);
  for (int t = 0; t < ntiles; t++) {
    const StPattern &T = tpat[(size_t)t];
    int              id = -1;
    const int        prev = t > 0 ? st.pid[(size_t)t - 1] : 0;
    if (!st.pats.empty()) {
      const StPattern &Q = st.pats[(size_t)prev];
      if (Q.L == T.L && !memcmp(Q.d, T.d, sizeof(int) * T.L) && !memcmp(Q.v, T.v, sizeof(double) * T.L)) id = prev;
    }
    for (int c = 0; c < (int)st.pats.size() && id < 0; c++) {
      const StPattern &Q = st.pats[(size_t)c];
      if (Q.L == T.L && !memcmp(Q.d, T.d, sizeof(int) * T.L) && !memcmp(Q.v, T.v, sizeof(double) * T.L)) id = c;
    }
    if (id < 0) {
      if ((int)st.pats.size() == PB_ST_MAXPAT) return 0;
      StPattern P = T;
      P.nwin = pattern_windows(P) + 1;
      id     = (int)st.pats.size();
      st.pats.push_back(P);
    }
    st.pid[(size_t)t] = (unsigned char)id;
  }
  st.nwin = 0;
  for (const StPattern &P : st.pats) st.nwin = std::max(st.nwin, P.nwin);
  // ghost entries: static schedule => thread k owns a contiguous, ascending range of tiles: concatenation is already sorted by row
  for (const OffDiagEntries &e : toff) {
    off.row.insert(off.row.end(), e.row.begin(), e.row.end());
    off.gcol.insert(off.gcol.end(), e.gcol.begin(), e.gcol.end());
    off.val.insert(off.val.end(), e.val.begin(), e.val.end());
  }
  nnz_diag = nd;
  st.valid = true;
  return 0;
}

}   // namespace pb
