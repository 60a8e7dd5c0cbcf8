// caar_dss.cu — HOMME's direct stiffness summation (edgeVpack / bndry_exchangeV / edgeVunpack, then rspheremp) on the
// handle's elements, and neighbor_minmax of the tracer limiter bounds, both over the element connectivity of
// caar_set_connectivity. The operations are specified in include/caar_b200.h; the kernels restate them operation for
// operation (every operation rounded separately, sums sequential in copy order), so their results are bit-reproducible
// and equal the FP64 restatement of tests/dss_oracle.py.
//
// Tables (built once on the host, build_dss_tables): the copies of every point, i.e. the (e, p) with one global id, are
// sorted by (e, p); the first is the point's owner. Groups are stored in the order of their owners, so the walk goes
// element by element: start[g] .. start[g+1] index copy[], each copy packed as e*16 + p. Every (e, p) is in exactly one
// group, so copy[] has 16 E entries.
//
// dss_kernel: one thread per group, grid-stride over the groups in owner order. The thread loads its copy indices and
// spheremp values once, forms m and r = 1/m, then walks the selected fields and the levels, reading every copy, summing
// in copy order and writing S*r to every copy. In place in one launch, without atomics or an edge buffer: every value
// (e, p, field, level) is read and written by the one thread that owns the group of (e, p), and by no other thread, so
// no thread ever reads a value another thread has written, whatever the order in which the threads run. The same holds
// inside a thread, whose loads of a batch of levels all precede its stores of that batch, at disjoint addresses.
// Groups of up to 4 copies (every group of a cubed sphere) keep their indices in registers; larger groups take a loop
// that reads the indices from the table per level.
//
// neighbor_minmax_kernel: one thread per (e, iq, k) bound pair of the whole array, k fastest, so that a warp reads one
// contiguous row of each neighbour. It reads the old bounds and writes a second array (the caller swaps the two), so
// the result does not depend on the order in which threads run; tracers iq >= qsize are copied.
//
// Across partitioned handles (caar_set_partition; tables and buffer layout at HaloHostTables in caar_device.cuh):
// dss_pack_kernel writes one record per boundary copy for the other parts; dss_unpack_kernel is dss_kernel's walk in
// which groups with remote copies read those copies from the received records; neighbor_minmax_pack_kernel and
// neighbor_minmax_unpack_kernel do the same with the bound rows of boundary elements. caar_dss_interior runs dss_kernel on
// the local groups without remote copies; caar_dss_boundary runs dss_boundary_kernel, one thread per (group with a
// remote copy, slice, batch of levels), on the others.
#include <algorithm>
#include <cstring>
#include <vector>

#include "caar_device.cuh"

namespace caar {

namespace {

constexpr int DSS_THREADS = 256;
constexpr int DSS_CTAS_PER_SM = 2;  // 512 threads per SM (128 registers), each with a batch of levels of every copy in flight
constexpr int FAST_COPIES = 4;      // the largest group of a cubed sphere

// The selected fields as up to 4 runs of slices: run i is count[i] slices, step[i] doubles apart from base[i] on, each a
// [L][16][w[i]] block in every element's block of estride[i] doubles (dp3d, v, T at tl; Qdp(qtl) of tracers < qsize)
struct DssArgs {
  double* base[4];
  size_t estride[4], step[4];
  int w[4], count[4];
  int nruns;
  const double* spheremp;    // [E][16]
  const int* start;          // [ngroups + 1]
  const int* copy;           // [16 E], e*16 + p
  int ngroups, L;
};

// W doubles per point: 1 for scalars, 2 for the two components of v (each its own scalar field)
template <int W>
__device__ __forceinline__ void load(const double* p, double (&o)[W]) {
  if constexpr (W == 2) {
    const double2 t = *reinterpret_cast<const double2*>(p);
    o[0] = t.x;
    o[1] = t.y;
  } else {
    o[0] = *p;
  }
}
template <int W>
__device__ __forceinline__ void store(double* p, const double (&o)[W]) {
  if constexpr (W == 2) *reinterpret_cast<double2*>(p) = make_double2(o[0], o[1]);
  else *p = o[0];
}

// One group: its copies copy[c0 .. c0+n) and r = 1/m; for n <= FAST_COPIES also the copies and their spheremp values
struct Group {
  int c0, n;
  int cp[FAST_COPIES];
  double s[FAST_COPIES];
  double r;
};

// One field slice of one group: every level, every component. `base` is the slice in element 0 and every element's block
// is `estride` doubles. Groups of up to FAST_COPIES copies take the levels in batches of 4 / W with all loads of a batch
// first; larger groups re-read their copies from the table for every level.
template <int W, bool PROJECT>
__device__ __forceinline__ void dss_slice(double* base, size_t estride, const DssArgs& A, const Group& g) {
  const int L = A.L;
  if (g.n <= FAST_COPIES) {
    constexpr int LV = 4 / W;
    double* q[FAST_COPIES];
#pragma unroll
    for (int c = 0; c < FAST_COPIES; ++c) q[c] = base + (size_t)(g.cp[c] >> 4) * estride + (g.cp[c] & 15) * W;
#pragma unroll 1
    for (int k0 = 0; k0 < L; k0 += LV) {
      double f[LV][FAST_COPIES][W];
#pragma unroll
      for (int j = 0; j < LV; ++j)
#pragma unroll
        for (int c = 0; c < FAST_COPIES; ++c)
          if (k0 + j < L && c < g.n) load<W>(q[c] + (size_t)(k0 + j) * 16 * W, f[j][c]);
#pragma unroll
      for (int j = 0; j < LV; ++j) {
        if (k0 + j >= L) break;
        double out[W];
#pragma unroll
        for (int w = 0; w < W; ++w) {
          double S = PROJECT ? __dmul_rn(g.s[0], f[j][0][w]) : f[j][0][w];
#pragma unroll
          for (int c = 1; c < FAST_COPIES; ++c)
            if (c < g.n) S = __dadd_rn(S, PROJECT ? __dmul_rn(g.s[c], f[j][c][w]) : f[j][c][w]);
          out[w] = __dmul_rn(S, g.r);
        }
#pragma unroll
        for (int c = 0; c < FAST_COPIES; ++c)
          if (c < g.n) store<W>(q[c] + (size_t)(k0 + j) * 16 * W, out);
      }
    }
    return;
  }
#pragma unroll 1
  for (int k = 0; k < L; ++k) {
    double S[W];
#pragma unroll 1
    for (int c = 0; c < g.n; ++c) {
      const int cp = A.copy[g.c0 + c];
      double f[W];
      load<W>(base + (size_t)(cp >> 4) * estride + (size_t)k * 16 * W + (cp & 15) * W, f);
      const double s = PROJECT ? A.spheremp[cp] : 0.0;
#pragma unroll
      for (int w = 0; w < W; ++w) {
        const double t = PROJECT ? __dmul_rn(s, f[w]) : f[w];
        S[w] = c == 0 ? t : __dadd_rn(S[w], t);
      }
    }
#pragma unroll
    for (int w = 0; w < W; ++w) S[w] = __dmul_rn(S[w], g.r);
#pragma unroll 1
    for (int c = 0; c < g.n; ++c) {
      const int cp = A.copy[g.c0 + c];
      store<W>(base + (size_t)(cp >> 4) * estride + (size_t)k * 16 * W + (cp & 15) * W, S);
    }
  }
}

// One group: the spheremp of its copies, m, r, then every selected slice; g.c0, g.n and g.cp (the first FAST_COPIES
// copies, the first one repeated beyond g.n) are set, and every copy is local
template <bool PROJECT>
__device__ __forceinline__ void dss_group(const DssArgs& A, Group& g) {
#pragma unroll
  for (int c = 0; c < FAST_COPIES; ++c) g.s[c] = A.spheremp[g.cp[c]];
  double m = g.s[0];
#pragma unroll
  for (int c = 1; c < FAST_COPIES; ++c)
    if (c < g.n) m = __dadd_rn(m, g.s[c]);
  for (int c = FAST_COPIES; c < g.n; ++c) m = __dadd_rn(m, A.spheremp[A.copy[g.c0 + c]]);
  g.r = __ddiv_rn(1.0, m);
#pragma unroll 1
  for (int run = 0; run < A.nruns; ++run)
#pragma unroll 1
    for (int j = 0; j < A.count[run]; ++j) {
      double* base = A.base[run] + j * A.step[run];
      if (A.w[run] == 2) dss_slice<2, PROJECT>(base, A.estride[run], A, g);
      else dss_slice<1, PROJECT>(base, A.estride[run], A, g);
    }
}

template <bool PROJECT>
__global__ void __launch_bounds__(DSS_THREADS, DSS_CTAS_PER_SM) dss_kernel(const DssArgs A) {
  for (size_t i = (size_t)blockIdx.x * DSS_THREADS + threadIdx.x; i < (size_t)A.ngroups;
       i += (size_t)gridDim.x * DSS_THREADS) {
    Group g;
    g.c0 = A.start[i];
    g.n = A.start[i + 1] - g.c0;
#pragma unroll
    for (int c = 0; c < FAST_COPIES; ++c) g.cp[c] = A.copy[g.c0 + (c < g.n ? c : 0)];
    dss_group<PROJECT>(A, g);
  }
}

// ---- the exchange between partitioned handles ----
// A DSS buffer (HaloTables): record R, in the segment seg[R] = {first record, records}, holds value v at
// buf[first * nv + v * records + R - first]
struct HaloArgs {
  double* buf;      // the send buffer (pack) or the receive buffer (unpack)
  const int2* seg;  // [records]
  const int* copy;  // pack: the local copy e*16 + p of every record
  int nrec, nv;
};

__device__ __forceinline__ double* record(const HaloArgs& H, int R, size_t* stride) {
  const int2 sg = H.seg[R];
  *stride = (size_t)sg.y;
  return H.buf + (size_t)sg.x * H.nv + (R - sg.x);
}

// One thread per send record: spheremp, then the selected slices level by level, each batch of values loaded before
// it is stored. Consecutive records are consecutive doubles of every value row, so the stores of a warp coalesce.
__global__ void __launch_bounds__(DSS_THREADS) dss_pack_kernel(const DssArgs A, const HaloArgs H) {
  constexpr int LV = 8;
  for (int R = blockIdx.x * DSS_THREADS + threadIdx.x; R < H.nrec; R += gridDim.x * DSS_THREADS) {
    const int cp = H.copy[R];
    size_t st;
    double* o = record(H, R, &st);
    o[0] = A.spheremp[cp];
    o += st;
#pragma unroll 1
    for (int run = 0; run < A.nruns; ++run)
#pragma unroll 1
      for (int j = 0; j < A.count[run]; ++j) {
        const int W = A.w[run];
        const double* p = A.base[run] + j * A.step[run] + (size_t)(cp >> 4) * A.estride[run] + (cp & 15) * W;
        const int n = A.L * W;  // value v = k*W + w of the slice is p[k * 16 W + w]
#pragma unroll 1
        for (int v0 = 0; v0 < n; v0 += LV) {
          double f[LV];
#pragma unroll
          for (int i = 0; i < LV; ++i)
            if (v0 + i < n) f[i] = p[(size_t)((v0 + i) / W) * 16 * W + (v0 + i) % W];
#pragma unroll
          for (int i = 0; i < LV; ++i)
            if (v0 + i < n) o[(size_t)(v0 + i) * st] = f[i];
        }
        o += (size_t)n * st;
      }
  }
}

// One slice of a group with remote copies: dss_slice's general loop, with a remote copy's value v0 + k*W + w and its
// spheremp read from its record; only the local copies are written
template <int W, bool PROJECT>
__device__ __forceinline__ void dss_slice_halo(double* base, size_t estride, const DssArgs& A, const HaloArgs& H,
                                               const Group& g, int v0) {
#pragma unroll 1
  for (int k = 0; k < A.L; ++k) {
    double S[W];
#pragma unroll 1
    for (int c = 0; c < g.n; ++c) {
      const int cp = A.copy[g.c0 + c];
      double f[W], s;
      if (cp >= 0) {
        load<W>(base + (size_t)(cp >> 4) * estride + (size_t)k * 16 * W + (cp & 15) * W, f);
        s = PROJECT ? A.spheremp[cp] : 0.0;
      } else {
        size_t st;
        const double* o = record(H, -1 - cp, &st);
#pragma unroll
        for (int w = 0; w < W; ++w) f[w] = o[(size_t)(v0 + k * W + w) * st];
        s = PROJECT ? o[0] : 0.0;
      }
#pragma unroll
      for (int w = 0; w < W; ++w) {
        const double t = PROJECT ? __dmul_rn(s, f[w]) : f[w];
        S[w] = c == 0 ? t : __dadd_rn(S[w], t);
      }
    }
#pragma unroll
    for (int w = 0; w < W; ++w) S[w] = __dmul_rn(S[w], g.r);
#pragma unroll 1
    for (int c = 0; c < g.n; ++c) {
      const int cp = A.copy[g.c0 + c];
      if (cp >= 0) store<W>(base + (size_t)(cp >> 4) * estride + (size_t)k * 16 * W + (cp & 15) * W, S);
    }
  }
}

// dss_kernel's walk over the groups of HaloTables. A group whose copies are all local takes dss_kernel's path, so that
// without remote copies the result is caar_dss's bit for bit; a group with remote copies takes the general loop. In
// place as dss_kernel: a local value is read and written by the thread of its group only, and the receive buffer is
// only read.
template <bool PROJECT>
__global__ void __launch_bounds__(DSS_THREADS, DSS_CTAS_PER_SM) dss_unpack_kernel(const DssArgs A, const HaloArgs H) {
  for (size_t i = (size_t)blockIdx.x * DSS_THREADS + threadIdx.x; i < (size_t)A.ngroups;
       i += (size_t)gridDim.x * DSS_THREADS) {
    Group g;
    g.c0 = A.start[i];
    g.n = A.start[i + 1] - g.c0;
    bool local = true;
#pragma unroll
    for (int c = 0; c < FAST_COPIES; ++c) {
      g.cp[c] = A.copy[g.c0 + (c < g.n ? c : 0)];
      local = local && g.cp[c] >= 0;
    }
    for (int c = FAST_COPIES; c < g.n; ++c) local = local && A.copy[g.c0 + c] >= 0;
    if (local) {
      dss_group<PROJECT>(A, g);
      continue;
    }
    double m = 0.0;
#pragma unroll 1
    for (int c = 0; c < g.n; ++c) {
      const int cp = A.copy[g.c0 + c];
      size_t st;
      const double s = cp >= 0 ? A.spheremp[cp] : record(H, -1 - cp, &st)[0];
      m = c == 0 ? s : __dadd_rn(m, s);
    }
    g.r = __ddiv_rn(1.0, m);
    int v0 = 1;
#pragma unroll 1
    for (int run = 0; run < A.nruns; ++run)
#pragma unroll 1
      for (int j = 0; j < A.count[run]; ++j) {
        double* base = A.base[run] + j * A.step[run];
        if (A.w[run] == 2) dss_slice_halo<2, PROJECT>(base, A.estride[run], A, H, g, v0);
        else dss_slice_halo<1, PROJECT>(base, A.estride[run], A, H, g, v0);
        v0 += A.L * A.w[run];
      }
  }
}

// ---- the boundary groups alone (caar_dss_boundary) ----
constexpr int BATCH = 4;  // levels per thread of dss_boundary_kernel: 18 batches at nlev 72

// Levels k0 .. k0+BATCH (clipped to L) of one slice of the boundary group copy[c0 .. c0+n): m and r in copy order,
// then, per level, every copy (local from the field, remote from its record, value v0 + k*W + w) summed in copy order;
// only the local copies are written. The operations and their order are dss_unpack_kernel's for a group with remote
// copies, so the bits are too. Groups of up to FAST_COPIES copies load the whole batch before any store.
template <int W, bool PROJECT>
__device__ __forceinline__ void boundary_batch(double* base, size_t estride, const DssArgs& A, const HaloArgs& H,
                                               int c0, int n, int v0, int k0) {
  const int nk = min(BATCH, A.L - k0);
  if (n <= FAST_COPIES) {
    double* p[FAST_COPIES];  // level k0 of the copy
    int ws[FAST_COPIES];     // doubles between components: 1 for a local copy, its segment's records for a remote one
    double s[FAST_COPIES];
    bool loc[FAST_COPIES];
#pragma unroll
    for (int c = 0; c < FAST_COPIES; ++c) {
      const int cp = A.copy[c0 + (c < n ? c : 0)];
      loc[c] = cp >= 0;
      if (loc[c]) {
        p[c] = base + (size_t)(cp >> 4) * estride + (size_t)k0 * 16 * W + (cp & 15) * W;
        ws[c] = 1;
        s[c] = A.spheremp[cp];
      } else {
        size_t st;
        double* o = record(H, -1 - cp, &st);
        p[c] = o + (size_t)(v0 + k0 * W) * st;
        ws[c] = (int)st;
        s[c] = o[0];
      }
    }
    double m = s[0];
#pragma unroll
    for (int c = 1; c < FAST_COPIES; ++c)
      if (c < n) m = __dadd_rn(m, s[c]);
    const double r = __ddiv_rn(1.0, m);
    constexpr int LV = BATCH / W;  // levels in flight: 4 values of every copy, as in dss_slice
#pragma unroll 1
    for (int j0 = 0; j0 < nk; j0 += LV) {
      double f[LV][FAST_COPIES][W];
#pragma unroll
      for (int j = 0; j < LV; ++j)
#pragma unroll
        for (int c = 0; c < FAST_COPIES; ++c)
          if (j0 + j < nk && c < n) {
            const double* q = p[c] + (size_t)(j0 + j) * (loc[c] ? 16 * W : W * ws[c]);
            if (loc[c]) {
              load<W>(q, f[j][c]);
            } else {
#pragma unroll
              for (int w = 0; w < W; ++w) f[j][c][w] = q[(size_t)w * ws[c]];
            }
          }
#pragma unroll
      for (int j = 0; j < LV; ++j) {
        if (j0 + j >= nk) break;
        double out[W];
#pragma unroll
        for (int w = 0; w < W; ++w) {
          double S = PROJECT ? __dmul_rn(s[0], f[j][0][w]) : f[j][0][w];
#pragma unroll
          for (int c = 1; c < FAST_COPIES; ++c)
            if (c < n) S = __dadd_rn(S, PROJECT ? __dmul_rn(s[c], f[j][c][w]) : f[j][c][w]);
          out[w] = __dmul_rn(S, r);
        }
#pragma unroll
        for (int c = 0; c < FAST_COPIES; ++c)
          if (c < n && loc[c]) store<W>(p[c] + (size_t)(j0 + j) * 16 * W, out);
      }
    }
    return;
  }
  double m = 0.0;
#pragma unroll 1
  for (int c = 0; c < n; ++c) {
    const int cp = A.copy[c0 + c];
    size_t st;
    const double s = cp >= 0 ? A.spheremp[cp] : record(H, -1 - cp, &st)[0];
    m = c == 0 ? s : __dadd_rn(m, s);
  }
  const double r = __ddiv_rn(1.0, m);
#pragma unroll 1
  for (int k = k0; k < k0 + nk; ++k) {  // dss_slice_halo's level loop over this batch
    double S[W];
#pragma unroll 1
    for (int c = 0; c < n; ++c) {
      const int cp = A.copy[c0 + c];
      double f[W], s;
      if (cp >= 0) {
        load<W>(base + (size_t)(cp >> 4) * estride + (size_t)k * 16 * W + (cp & 15) * W, f);
        s = PROJECT ? A.spheremp[cp] : 0.0;
      } else {
        size_t st;
        const double* o = record(H, -1 - cp, &st);
#pragma unroll
        for (int w = 0; w < W; ++w) f[w] = o[(size_t)(v0 + k * W + w) * st];
        s = PROJECT ? o[0] : 0.0;
      }
#pragma unroll
      for (int w = 0; w < W; ++w) {
        const double t = PROJECT ? __dmul_rn(s, f[w]) : f[w];
        S[w] = c == 0 ? t : __dadd_rn(S[w], t);
      }
    }
#pragma unroll
    for (int w = 0; w < W; ++w) S[w] = __dmul_rn(S[w], r);
#pragma unroll 1
    for (int c = 0; c < n; ++c) {
      const int cp = A.copy[c0 + c];
      if (cp >= 0) store<W>(base + (size_t)(cp >> 4) * estride + (size_t)k * 16 * W + (cp & 15) * W, S);
    }
  }
}

// One thread per (boundary group, selected slice, batch of BATCH levels), the group fastest, so that a warp walks
// neighbouring points of one element and consecutive records. In place without atomics: every (local copy, slice,
// level) is read and written by one thread, and the receive buffer is only read.
template <bool PROJECT>
__global__ void __launch_bounds__(DSS_THREADS, DSS_CTAS_PER_SM) dss_boundary_kernel(const DssArgs A, const HaloArgs H,
                                                                                     int nslices) {
  const int nbatch = (A.L + BATCH - 1) / BATCH;
  const size_t total = (size_t)A.ngroups * nslices * nbatch;
  for (size_t i = (size_t)blockIdx.x * DSS_THREADS + threadIdx.x; i < total; i += (size_t)gridDim.x * DSS_THREADS) {
    const int g = (int)(i % A.ngroups);
    const size_t rest = i / A.ngroups;
    const int k0 = (int)(rest % nbatch) * BATCH;
    int j = (int)(rest / nbatch), run = 0, v0 = 1;  // slice j -> run, slice within the run, first value of its record
    while (j >= A.count[run]) {
      v0 += A.count[run] * A.L * A.w[run];
      j -= A.count[run];
      ++run;
    }
    v0 += j * A.L * A.w[run];
    double* base = A.base[run] + j * A.step[run];
    const int c0 = A.start[g], n = A.start[g + 1] - c0;
    if (A.w[run] == 2) boundary_batch<2, PROJECT>(base, A.estride[run], A, H, c0, n, v0, k0);
    else boundary_batch<1, PROJECT>(base, A.estride[run], A, H, c0, n, v0, k0);
  }
}

// neighbor_minmax of bound pair i; with HALO a neighbour q >= nelem is row q - nelem of rin, rrow pairs apart
template <bool HALO>
__device__ __forceinline__ double2 minmax_pair(const double2* __restrict__ in, const int* __restrict__ nb_start,
                                               const int* __restrict__ nb, size_t i, int row, int L, int qsize,
                                               const double2* __restrict__ rin, int nelem, int rrow) {
  const int e = (int)(i / row), o = (int)(i - (size_t)e * row);
  double2 b = in[i];
  if (o / L < qsize)
    for (int j = nb_start[e]; j < nb_start[e + 1]; ++j) {
      const int q = nb[j];
      const double2 t = (!HALO || q < nelem) ? in[(size_t)q * row + o] : rin[(size_t)(q - nelem) * rrow + o];
      if (t.x < b.x) b.x = t.x;
      if (t.y > b.y) b.y = t.y;
    }
  return b;
}

__global__ void __launch_bounds__(DSS_THREADS) neighbor_minmax_kernel(const double2* __restrict__ in,
                                                                      double2* __restrict__ out,
                                                                      const int* __restrict__ nb_start,
                                                                      const int* __restrict__ nb, size_t n, int row,
                                                                      int L, int qsize) {
  // row = qsize_d * L bound pairs per element
  for (size_t i = (size_t)blockIdx.x * DSS_THREADS + threadIdx.x; i < n; i += (size_t)gridDim.x * DSS_THREADS)
    out[i] = minmax_pair<false>(in, nb_start, nb, i, row, L, qsize, nullptr, 0, 0);
}

// neighbor_minmax_kernel with received rows of qsize * L pairs
__global__ void __launch_bounds__(DSS_THREADS) neighbor_minmax_unpack_kernel(
    const double2* __restrict__ in, double2* __restrict__ out, const int* __restrict__ nb_start,
    const int* __restrict__ nb, size_t n, int row, int L, int qsize, const double2* __restrict__ rin, int nelem) {
  for (size_t i = (size_t)blockIdx.x * DSS_THREADS + threadIdx.x; i < n; i += (size_t)gridDim.x * DSS_THREADS)
    out[i] = minmax_pair<true>(in, nb_start, nb, i, row, L, qsize, rin, nelem, qsize * L);
}

// one thread per (send row, pair): row R is the first rrow pairs of element el[R]
__global__ void __launch_bounds__(DSS_THREADS) neighbor_minmax_pack_kernel(const double2* __restrict__ in,
                                                                           double2* __restrict__ out,
                                                                           const int* __restrict__ el, size_t n,
                                                                           int row, int rrow) {
  for (size_t i = (size_t)blockIdx.x * DSS_THREADS + threadIdx.x; i < n; i += (size_t)gridDim.x * DSS_THREADS) {
    const size_t R = i / rrow;
    out[i] = in[(size_t)el[R] * row + (i - R * rrow)];
  }
}

// CTAs for `items` threads' work: one per DSS_THREADS items, at most one wave of at most max_per_sm CTAs per SM
template <typename Kernel>
unsigned grid_for(Kernel* k, size_t items, int max_per_sm, LaunchCache& cache, cudaError_t* e) {
  int per_sm = 1;
  *e = setup_launch(k, DSS_THREADS, 0, cache, &per_sm);
  size_t blocks = (items + DSS_THREADS - 1) / DSS_THREADS;
  const size_t wave = (size_t)std::min(per_sm, max_per_sm) * sm_count();
  return (unsigned)std::min(blocks, wave);
}

bool selected(unsigned mask, int qsize) {
  return (mask & (CAAR_F_DP3D | CAAR_F_V | CAAR_F_T)) || ((mask & CAAR_F_QDP) && qsize > 0);
}

// the selected slices of caar_dss as runs, over the groups start / copy
DssArgs dss_args(const KernelArgs& a, unsigned mask, int tl, int qtl, int qsize, const int* start, const int* copy,
                 int ngroups) {
  DssArgs A;
  std::memset(&A, 0, sizeof A);
  const size_t lf = (size_t)a.nlev * 16;
  auto add = [&](double* base, size_t estride, int w, int count, size_t step) {
    A.base[A.nruns] = base;
    A.estride[A.nruns] = estride;
    A.w[A.nruns] = w;
    A.count[A.nruns] = count;
    A.step[A.nruns++] = step;
  };
  if (mask & CAAR_F_DP3D) add(a.dp3d + tl * lf, a.ntl * lf, 1, 1, 0);
  if (mask & CAAR_F_V) add(a.v + 2 * tl * lf, 2 * a.ntl * lf, 2, 1, 0);
  if (mask & CAAR_F_T) add(a.T + tl * lf, a.ntl * lf, 1, 1, 0);
  if ((mask & CAAR_F_QDP) && qsize > 0)  // Qdp is const in KernelArgs for the kernels that read it; this is the mirror
    add(const_cast<double*>(a.Qdp) + qtl * lf, 2 * a.qsize_d * lf, 1, qsize, 2 * lf);
  A.spheremp = a.spheremp;
  A.start = start;
  A.copy = copy;
  A.ngroups = ngroups;
  A.L = a.nlev;
  return A;
}

}  // namespace

int build_dss_tables(const long long* gid, int nelem, DssHostTables* t) {
  const size_t ncopy = (size_t)nelem * 16;
  struct Copy {
    long long gid;
    int cp;  // e*16 + p: (e, p) order
  };
  std::vector<Copy> c(ncopy);
  for (size_t i = 0; i < ncopy; ++i) c[i] = Copy{gid[i], (int)i};
  std::sort(c.begin(), c.end(), [](const Copy& a, const Copy& b) { return a.gid != b.gid ? a.gid < b.gid : a.cp < b.cp; });
  // groups = runs of one gid, each in (e, p) order; then in the order of their owners (first copies)
  std::vector<size_t> run;  // start of each run in c
  for (size_t i = 0; i < ncopy; ++i)
    if (i == 0 || c[i].gid != c[i - 1].gid) run.push_back(i);
  const size_t G = run.size();
  run.push_back(ncopy);
  std::vector<int> order(G);
  for (size_t g = 0; g < G; ++g) order[g] = (int)g;
  std::sort(order.begin(), order.end(), [&](int a, int b) { return c[run[a]].cp < c[run[b]].cp; });
  t->start.assign(G + 1, 0);
  t->copy.resize(ncopy);
  size_t k = 0;
  std::vector<long long> pairs;  // e * nelem + n for every two distinct elements that share a point
  for (size_t g = 0; g < G; ++g) {
    const size_t a = run[order[g]], b = run[order[g] + 1];
    t->start[g] = (int)k;
    for (size_t i = a; i < b; ++i) {
      t->copy[k++] = c[i].cp;
      for (size_t j = a; j < b; ++j) {
        const int ei = c[i].cp >> 4, ej = c[j].cp >> 4;
        if (ei != ej) pairs.push_back((long long)ei * nelem + ej);
      }
    }
  }
  t->start[G] = (int)k;
  std::sort(pairs.begin(), pairs.end());
  pairs.erase(std::unique(pairs.begin(), pairs.end()), pairs.end());
  t->nb_start.assign((size_t)nelem + 1, 0);
  t->nb.resize(pairs.size());
  for (size_t i = 0; i < pairs.size(); ++i) {
    t->nb[i] = (int)(pairs[i] % nelem);
    ++t->nb_start[pairs[i] / nelem + 1];
  }
  for (int e = 0; e < nelem; ++e) t->nb_start[e + 1] += t->nb_start[e];
  return (int)G;
}

void build_halo_tables(const long long* gid, int nelem_global, const int* part_start, int nparts, int part,
                       HaloHostTables* t) {
  const int e0 = part_start[part], nl = part_start[part + 1] - e0;
  const size_t ncopy = (size_t)nelem_global * 16;
  struct Copy {
    long long gid;
    int cp;  // global e*16 + p
  };
  std::vector<Copy> c(ncopy);
  for (size_t i = 0; i < ncopy; ++i) c[i] = Copy{gid[i], (int)i};
  std::sort(c.begin(), c.end(), [](const Copy& a, const Copy& b) { return a.gid != b.gid ? a.gid < b.gid : a.cp < b.cp; });
  auto part_of = [&](int ge) { return (int)(std::upper_bound(part_start, part_start + nparts + 1, ge) - part_start) - 1; };
  auto is_local = [&](int ge) { return ge >= e0 && ge < e0 + nl; };
  // the runs of one gid that hold a local copy; the remote copies of each (received, in global sort order per sender)
  // and the local copies for every other part that holds the point (sent, in the same order)
  std::vector<std::pair<size_t, size_t>> runs;
  std::vector<std::vector<size_t>> recv(nparts);
  std::vector<std::vector<int>> send(nparts);
  std::vector<long long> pairs;  // el * nelem_global + ge for local el and every other element ge that shares a point
  std::vector<int> parts;
  for (size_t a = 0, b; a < ncopy; a = b) {
    bool local = false;
    for (b = a; b < ncopy && c[b].gid == c[a].gid; ++b) local = local || is_local(c[b].cp >> 4);
    if (!local) continue;
    runs.emplace_back(a, b);
    parts.clear();
    for (size_t i = a; i < b; ++i) {
      const int gi = c[i].cp >> 4;
      if (!is_local(gi)) {
        const int q = part_of(gi);
        recv[q].push_back(i);
        if (std::find(parts.begin(), parts.end(), q) == parts.end()) parts.push_back(q);
        continue;
      }
      for (size_t j = a; j < b; ++j) {
        const int gj = c[j].cp >> 4;
        if (gj != gi) pairs.push_back((long long)(gi - e0) * nelem_global + gj);
      }
    }
    std::sort(parts.begin(), parts.end());
    for (int q : parts)
      for (size_t i = a; i < b; ++i)
        if (is_local(c[i].cp >> 4)) send[q].push_back(c[i].cp - e0 * 16);
  }
  for (auto& r : t->rec) r.assign((size_t)nparts + 1, 0);
  std::vector<int> rid(ncopy, -1);  // record of every received copy, by its place in c
  for (int q = 0; q < nparts; ++q) {
    t->rec[0][q + 1] = t->rec[0][q] + (int)send[q].size();
    t->rec[1][q + 1] = t->rec[1][q] + (int)recv[q].size();
    for (size_t k = 0; k < recv[q].size(); ++k) rid[recv[q][k]] = t->rec[1][q] + (int)k;
    t->send_copy.insert(t->send_copy.end(), send[q].begin(), send[q].end());
  }
  // the local groups in the order of their owners, every copy in global (e, p) order
  std::sort(runs.begin(), runs.end(), [&](const std::pair<size_t, size_t>& x, const std::pair<size_t, size_t>& y) {
    auto owner = [&](const std::pair<size_t, size_t>& r) {
      size_t i = r.first;
      while (!is_local(c[i].cp >> 4)) ++i;
      return c[i].cp;
    };
    return owner(x) < owner(y);
  });
  t->start.assign(1, 0);
  t->copy.clear();
  t->istart.assign(1, 0);
  t->icopy.clear();
  t->bstart.assign(1, 0);
  t->bcopy.clear();
  for (const auto& r : runs) {
    const size_t g0 = t->copy.size();
    for (size_t i = r.first; i < r.second; ++i)
      t->copy.push_back(is_local(c[i].cp >> 4) ? c[i].cp - e0 * 16 : -1 - rid[i]);
    t->start.push_back((int)t->copy.size());
    const bool interior = std::all_of(t->copy.begin() + g0, t->copy.end(), [](int cp) { return cp >= 0; });
    std::vector<int>& st = interior ? t->istart : t->bstart;
    std::vector<int>& cp = interior ? t->icopy : t->bcopy;
    cp.insert(cp.end(), t->copy.begin() + g0, t->copy.end());
    st.push_back((int)cp.size());
  }
  // neighbours: N(el) ascending by global element; a remote one is the row of its element among those received from
  // its part, which are the elements of that part with a neighbour here, ascending
  std::sort(pairs.begin(), pairs.end());
  pairs.erase(std::unique(pairs.begin(), pairs.end()), pairs.end());
  std::vector<std::vector<int>> send_el(nparts), recv_el(nparts);
  for (long long pr : pairs) {
    const int el = (int)(pr / nelem_global), gj = (int)(pr % nelem_global);
    if (is_local(gj)) continue;
    const int q = part_of(gj);
    recv_el[q].push_back(gj);
    if (send_el[q].empty() || send_el[q].back() != el) send_el[q].push_back(el);  // pairs ascend in el
  }
  for (int q = 0; q < nparts; ++q) {
    std::sort(recv_el[q].begin(), recv_el[q].end());
    recv_el[q].erase(std::unique(recv_el[q].begin(), recv_el[q].end()), recv_el[q].end());
    t->rec[2][q + 1] = t->rec[2][q] + (int)send_el[q].size();
    t->rec[3][q + 1] = t->rec[3][q] + (int)recv_el[q].size();
    t->send_el.insert(t->send_el.end(), send_el[q].begin(), send_el[q].end());
  }
  t->nb_start.assign((size_t)nl + 1, 0);
  t->nb.resize(pairs.size());
  for (size_t i = 0; i < pairs.size(); ++i) {
    const int el = (int)(pairs[i] / nelem_global), gj = (int)(pairs[i] % nelem_global);
    if (is_local(gj)) {
      t->nb[i] = gj - e0;
    } else {
      const int q = part_of(gj);
      const auto& r = recv_el[q];
      t->nb[i] = nl + t->rec[3][q] + (int)(std::lower_bound(r.begin(), r.end(), gj) - r.begin());
    }
    ++t->nb_start[el + 1];
  }
  for (int e = 0; e < nl; ++e) t->nb_start[e + 1] += t->nb_start[e];
}

size_t dss_record_doubles(unsigned mask, int qsize, int L) {
  if (!selected(mask, qsize)) return 0;
  const int per_level = !!(mask & CAAR_F_DP3D) + 2 * !!(mask & CAAR_F_V) + !!(mask & CAAR_F_T) +
                        ((mask & CAAR_F_QDP) ? qsize : 0);
  return 1 + (size_t)per_level * L;
}

namespace {

// dss_kernel over the groups start / copy: caar_dss, and the interior groups of a partitioned handle
cudaError_t launch_dss_groups(const KernelArgs& a, const int* start, const int* copy, int ngroups, unsigned mask,
                              int tl, int qtl, int qsize, int weighting, cudaStream_t s) {
  if (!selected(mask, qsize)) return cudaSuccess;
  const DssArgs A = dss_args(a, mask, tl, qtl, qsize, start, copy, ngroups);
  static LaunchCache cache[2];
  cudaError_t e = cudaSuccess;
  if (weighting == CAAR_DSS_PROJECT) {
    const unsigned grid = grid_for(dss_kernel<true>, (size_t)ngroups, DSS_CTAS_PER_SM, cache[1], &e);
    if (e != cudaSuccess) return e;
    dss_kernel<true><<<grid, DSS_THREADS, 0, s>>>(A);
  } else {
    const unsigned grid = grid_for(dss_kernel<false>, (size_t)ngroups, DSS_CTAS_PER_SM, cache[0], &e);
    if (e != cudaSuccess) return e;
    dss_kernel<false><<<grid, DSS_THREADS, 0, s>>>(A);
  }
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_dss(const KernelArgs& a, const DssTables& t, unsigned mask, int tl, int qtl, int qsize,
                       int weighting, cudaStream_t s) {
  return launch_dss_groups(a, t.start, t.copy, t.ngroups, mask, tl, qtl, qsize, weighting, s);
}

cudaError_t launch_dss_interior(const KernelArgs& a, const HaloTables& t, unsigned mask, int tl, int qtl, int qsize,
                                int weighting, cudaStream_t s) {
  if (t.ninterior == 0) return cudaSuccess;
  return launch_dss_groups(a, t.istart, t.icopy, t.ninterior, mask, tl, qtl, qsize, weighting, s);
}

cudaError_t launch_dss_boundary(const KernelArgs& a, const HaloTables& t, unsigned mask, int tl, int qtl, int qsize,
                                int weighting, cudaStream_t s) {
  if (!selected(mask, qsize) || t.nboundary == 0) return cudaSuccess;
  const DssArgs A = dss_args(a, mask, tl, qtl, qsize, t.bstart, t.bcopy, t.nboundary);
  const HaloArgs H{t.recv, t.recv_seg, nullptr, t.nrecv, (int)dss_record_doubles(mask, qsize, a.nlev)};
  int nslices = 0;
  for (int r = 0; r < A.nruns; ++r) nslices += A.count[r];
  const size_t items = (size_t)t.nboundary * nslices * ((a.nlev + BATCH - 1) / BATCH);
  static LaunchCache cache[2];
  cudaError_t e = cudaSuccess;
  if (weighting == CAAR_DSS_PROJECT) {
    const unsigned grid = grid_for(dss_boundary_kernel<true>, items, 2048 / DSS_THREADS, cache[1], &e);
    if (e != cudaSuccess) return e;
    dss_boundary_kernel<true><<<grid, DSS_THREADS, 0, s>>>(A, H, nslices);
  } else {
    const unsigned grid = grid_for(dss_boundary_kernel<false>, items, 2048 / DSS_THREADS, cache[0], &e);
    if (e != cudaSuccess) return e;
    dss_boundary_kernel<false><<<grid, DSS_THREADS, 0, s>>>(A, H, nslices);
  }
  return cudaGetLastError();
}

cudaError_t launch_neighbor_minmax(const DssTables& t, int nelem, int qsize_d, int L, int qsize, const double* in,
                                   double* out, cudaStream_t s) {
  if (qsize <= 0) return cudaSuccess;
  static LaunchCache cache;
  const size_t n = (size_t)nelem * qsize_d * L;
  cudaError_t e = cudaSuccess;
  const unsigned grid = grid_for(neighbor_minmax_kernel, n, 2048 / DSS_THREADS, cache, &e);
  if (e != cudaSuccess) return e;
  neighbor_minmax_kernel<<<grid, DSS_THREADS, 0, s>>>(reinterpret_cast<const double2*>(in),
                                                      reinterpret_cast<double2*>(out), t.nb_start, t.nb, n,
                                                      qsize_d * L, L, qsize);
  return cudaGetLastError();
}

cudaError_t launch_dss_pack(const KernelArgs& a, const HaloTables& t, unsigned mask, int tl, int qtl, int qsize,
                            cudaStream_t s) {
  if (!selected(mask, qsize) || t.nsend == 0) return cudaSuccess;
  const DssArgs A = dss_args(a, mask, tl, qtl, qsize, nullptr, nullptr, 0);
  const HaloArgs H{t.send, t.send_seg, t.send_copy, t.nsend, (int)dss_record_doubles(mask, qsize, a.nlev)};
  static LaunchCache cache;
  cudaError_t e = cudaSuccess;
  const unsigned grid = grid_for(dss_pack_kernel, (size_t)t.nsend, 2048 / DSS_THREADS, cache, &e);
  if (e != cudaSuccess) return e;
  dss_pack_kernel<<<grid, DSS_THREADS, 0, s>>>(A, H);
  return cudaGetLastError();
}

cudaError_t launch_dss_unpack(const KernelArgs& a, const HaloTables& t, unsigned mask, int tl, int qtl, int qsize,
                              int weighting, cudaStream_t s) {
  if (!selected(mask, qsize)) return cudaSuccess;
  const DssArgs A = dss_args(a, mask, tl, qtl, qsize, t.start, t.copy, t.ngroups);
  const HaloArgs H{t.recv, t.recv_seg, nullptr, t.nrecv, (int)dss_record_doubles(mask, qsize, a.nlev)};
  static LaunchCache cache[2];
  cudaError_t e = cudaSuccess;
  if (weighting == CAAR_DSS_PROJECT) {
    const unsigned grid = grid_for(dss_unpack_kernel<true>, (size_t)t.ngroups, DSS_CTAS_PER_SM, cache[1], &e);
    if (e != cudaSuccess) return e;
    dss_unpack_kernel<true><<<grid, DSS_THREADS, 0, s>>>(A, H);
  } else {
    const unsigned grid = grid_for(dss_unpack_kernel<false>, (size_t)t.ngroups, DSS_CTAS_PER_SM, cache[0], &e);
    if (e != cudaSuccess) return e;
    dss_unpack_kernel<false><<<grid, DSS_THREADS, 0, s>>>(A, H);
  }
  return cudaGetLastError();
}

cudaError_t launch_neighbor_minmax_pack(const HaloTables& t, int qsize_d, int L, int qsize, const double* bounds,
                                        cudaStream_t s) {
  const size_t n = (size_t)t.nsend_el * qsize * L;
  if (n == 0) return cudaSuccess;
  static LaunchCache cache;
  cudaError_t e = cudaSuccess;
  const unsigned grid = grid_for(neighbor_minmax_pack_kernel, n, 2048 / DSS_THREADS, cache, &e);
  if (e != cudaSuccess) return e;
  neighbor_minmax_pack_kernel<<<grid, DSS_THREADS, 0, s>>>(reinterpret_cast<const double2*>(bounds),
                                                           reinterpret_cast<double2*>(t.send), t.send_el, n,
                                                           qsize_d * L, qsize * L);
  return cudaGetLastError();
}

cudaError_t launch_neighbor_minmax_unpack(const HaloTables& t, int nelem, int qsize_d, int L, int qsize,
                                          const double* in, double* out, cudaStream_t s) {
  if (qsize <= 0) return cudaSuccess;
  static LaunchCache cache;
  const size_t n = (size_t)nelem * qsize_d * L;
  cudaError_t e = cudaSuccess;
  const unsigned grid = grid_for(neighbor_minmax_unpack_kernel, n, 2048 / DSS_THREADS, cache, &e);
  if (e != cudaSuccess) return e;
  neighbor_minmax_unpack_kernel<<<grid, DSS_THREADS, 0, s>>>(
      reinterpret_cast<const double2*>(in), reinterpret_cast<double2*>(out), t.nb_start, t.nb, n, qsize_d * L, L,
      qsize, reinterpret_cast<const double2*>(t.recv), nelem);
  return cudaGetLastError();
}

}  // namespace caar
