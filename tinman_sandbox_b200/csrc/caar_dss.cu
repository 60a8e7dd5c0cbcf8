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

template <bool PROJECT>
__global__ void __launch_bounds__(DSS_THREADS, DSS_CTAS_PER_SM) dss_kernel(const DssArgs A) {
  for (size_t i = (size_t)blockIdx.x * DSS_THREADS + threadIdx.x; i < (size_t)A.ngroups;
       i += (size_t)gridDim.x * DSS_THREADS) {
    Group g;
    g.c0 = A.start[i];
    g.n = A.start[i + 1] - g.c0;
#pragma unroll
    for (int c = 0; c < FAST_COPIES; ++c) {
      g.cp[c] = A.copy[g.c0 + (c < g.n ? c : 0)];
      g.s[c] = A.spheremp[g.cp[c]];
    }
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
}

__global__ void __launch_bounds__(DSS_THREADS) neighbor_minmax_kernel(const double2* __restrict__ in,
                                                                      double2* __restrict__ out,
                                                                      const int* __restrict__ nb_start,
                                                                      const int* __restrict__ nb, size_t n, int row,
                                                                      int L, int qsize) {
  // row = qsize_d * L bound pairs per element
  for (size_t i = (size_t)blockIdx.x * DSS_THREADS + threadIdx.x; i < n; i += (size_t)gridDim.x * DSS_THREADS) {
    const int e = (int)(i / row), o = (int)(i - (size_t)e * row);
    double2 b = in[i];
    if (o / L < qsize)
      for (int j = nb_start[e]; j < nb_start[e + 1]; ++j) {
        const double2 t = in[(size_t)nb[j] * row + o];
        if (t.x < b.x) b.x = t.x;
        if (t.y > b.y) b.y = t.y;
      }
    out[i] = b;
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

cudaError_t launch_dss(const KernelArgs& a, const DssTables& t, unsigned mask, int tl, int qtl, int qsize,
                       int weighting, cudaStream_t s) {
  if (!(mask & (CAAR_F_DP3D | CAAR_F_V | CAAR_F_T)) && !((mask & CAAR_F_QDP) && qsize > 0)) return cudaSuccess;
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
  A.start = t.start;
  A.copy = t.copy;
  A.ngroups = t.ngroups;
  A.L = a.nlev;
  static LaunchCache cache[2];
  cudaError_t e = cudaSuccess;
  if (weighting == CAAR_DSS_PROJECT) {
    const unsigned grid = grid_for(dss_kernel<true>, (size_t)t.ngroups, DSS_CTAS_PER_SM, cache[1], &e);
    if (e != cudaSuccess) return e;
    dss_kernel<true><<<grid, DSS_THREADS, 0, s>>>(A);
  } else {
    const unsigned grid = grid_for(dss_kernel<false>, (size_t)t.ngroups, DSS_CTAS_PER_SM, cache[0], &e);
    if (e != cudaSuccess) return e;
    dss_kernel<false><<<grid, DSS_THREADS, 0, s>>>(A);
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

}  // namespace caar
