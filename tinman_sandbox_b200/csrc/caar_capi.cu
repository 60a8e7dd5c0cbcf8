// caar_capi.cu — the C-ABI of include/caar_b200.h over the CUDA kernels. No CPU fallback: every
// compute entry point needs a CUDA device and fails with CAAR_ERR_CUDA otherwise.
#include <cstdarg>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <new>

#include "caar_device.cuh"

#ifndef CAAR_HOST_DEFAULT_ZERO_COPY
#define CAAR_HOST_DEFAULT_ZERO_COPY 0  // chunk_elems == 0 uses the staged pipeline unless CAAR_HOST_PATH=zerocopy
#endif

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
  return code;
}

#define CU_TRY(expr)                                                                          \
  do {                                                                                        \
    cudaError_t e_ = (expr);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return fail(e_ == cudaErrorMemoryAllocation ? CAAR_ERR_NOMEM : CAAR_ERR_CUDA,           \
                  "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

size_t field_count(const caar_dims& d, int f) {
  const size_t E = (size_t)d.nelem, L = (size_t)d.nlev, P = 16;
  switch (f) {
    case 0: case 1: return E * P * 4;
    case 2: case 3: case 4: case 5: case 9: return E * P;
    case 6: case 8: return E * d.ntl * L * P;
    case 7: return E * d.ntl * L * P * 2;
    case 10: return E * d.qsize_d * 2 * L * P;
    case 11: return E * (L + 1) * P;
    case 12: case 13: case 14: return E * L * P;
    case 15: return E * L * P * 2;
  }
  return 0;
}

double* const* as_table(const caar_arrays* a) { return reinterpret_cast<double* const*>(a); }

}  // namespace

struct caar_handle_s {
  caar_dims dims;
  int device;
  cudaStream_t own_stream, stream;
  double* dev[CAAR_NUM_FIELDS];
  bool params_set;
  caar_constants c;
  double dvv[16], ps0, hyai0;
  double* partial;    // [nelem][16] device: norms use [nelem][3], checksums [nelem][8][2]
  unsigned long long* bits;  // [nelem][7] device (checksums)
  double* out3;       // [16 doubles + 7 u64] device: results of the norm / checksum reductions
  double* out3_host;  // the same, pinned
  cudaEvent_t ev0, ev1;
  long long launches;
  caar::TmaMaps* tma;  // TMA descriptors of the device mirrors (nlev with a TMA-pipelined kernel only)
  // caar_run_host pipeline: copy-in and copy-out streams, two events per element chunk (grown on demand)
  cudaStream_t s_in, s_in2, s_out;  // s_in2: second copy-in stream (CAAR_HOST_IN_STREAMS=2)
  cudaEvent_t* chunk_ev;
  int n_chunk_ev;
  cudaEvent_t ev_fence;
  // caar_run_host zero-copy path: TMA descriptors over the caller's mapped host arrays, rebuilt when they move
  int rsplit;        // > 0 vertically Lagrangian (default 1), 0 Eulerian
  double* hybi_dev;  // [nlev+1], Eulerian branch only
  double* extra[5];  // arrays beyond struct Arrays: vstar, qtens, tensorVisc, scalar in / out (allocated on first use)
  double* stage;  // device staging buffer of the Fortran-layout copies (allocated on first use)
  // device [2]: the tile scheduler of the thread-per-level laplacians (next chunk, warps done), zero between launches.
  // One pair per handle: all launches of a handle are ordered on its stream, so no two of them share it.
  unsigned* lapflat_sched;
  caar::TmaMaps* tma_host;
  double* tma_host_key[CAAR_NUM_FIELDS];
};

static_assert(sizeof(caar_arrays) == CAAR_NUM_FIELDS * sizeof(double*), "caar_arrays must be 16 pointers");
// Layouts that include/caar_b200.f90 (bind(C) derived types) and the ctypes binding assume
static_assert(sizeof(caar_dims) == 20 && offsetof(caar_dims, nlev) == 4 && offsetof(caar_dims, ntl) == 16, "caar_dims: 5 ints");
static_assert(offsetof(caar_arrays, elem_state_dp3d) == 48 && offsetof(caar_arrays, elem_derived_vn0) == 120,
              "caar_arrays: the order of struct Arrays");
static_assert(sizeof(caar_constants) == 48 && offsetof(caar_constants, kappa) == 40, "caar_constants: 6 doubles");
static_assert(sizeof(caar_control) == 32 && offsetof(caar_control, qn0) == 20 && offsetof(caar_control, dt2) == 24,
              "caar_control: 6 ints + 1 double");
static_assert(sizeof(caar_checksum) == 184 && offsetof(caar_checksum, sumsq) == 56 && offsetof(caar_checksum, bits) == 112 &&
                  offsetof(caar_checksum, energy) == 168,
              "caar_checksum: 7 + 7 doubles, 7 64-bit integers, 2 doubles");

namespace {

struct DeviceGuard {
  int prev;
  bool ok;
  explicit DeviceGuard(int dev) : prev(-1), ok(false) {
    if (cudaGetDevice(&prev) != cudaSuccess) return;
    ok = (cudaSetDevice(dev) == cudaSuccess);
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

int validate_control(const caar_handle_s* h, const caar_control* ctl) {
  const caar_dims& d = h->dims;
  if (!ctl) return fail(CAAR_ERR_INVALID, "control is null");
  if (ctl->nets < 0 || ctl->nete > d.nelem || ctl->nets > ctl->nete)
    return fail(CAAR_ERR_INVALID, "element range [%d,%d) outside [0,%d)", ctl->nets, ctl->nete, d.nelem);
  const int tl[3] = {ctl->n0, ctl->np1, ctl->nm1};
  for (int i = 0; i < 3; ++i)
    if (tl[i] < 0 || tl[i] >= d.ntl) return fail(CAAR_ERR_INVALID, "time level %d outside [0,%d)", tl[i], d.ntl);
  if (ctl->qn0 < -1 || ctl->qn0 >= 2) return fail(CAAR_ERR_INVALID, "qn0=%d must be -1, 0 or 1", ctl->qn0);
  return CAAR_OK;
}

// the fused kernels cover the vertically Lagrangian branch, and the Eulerian one where launch_fused says so;
// everything else runs on the generic reference-order kernel (still on the GPU)
bool uses_fused(const caar_handle_s* h, int mode) {
  const bool fused = mode == CAAR_MODE_FAST && caar::fused_supports(h->dims.nlev) &&
                     (h->rsplit > 0 || caar::fused_supports_eulerian(h->dims.nlev));
  if (mode == CAAR_MODE_FAST && !fused) {  // never silent: the reference-order kernel is ~6x slower
    static bool told = false;
    if (!told) {
      told = true;
      fprintf(stderr, "[caar] CAAR_MODE_FAST: no fused kernel instance for nlev=%d (instances cover nlev <= 128); "
                      "running the reference-order kernel instead (see caar_describe)\n", h->dims.nlev);
    }
  }
  return fused;
}
// eta_dot_dpdn travels when the kernel really updates it: the reference-order kernel always does (+= 0 included),
// the fused kernels only on the Eulerian branch
bool moves_eta(const caar_handle_s* h, int mode) { return !uses_fused(h, mode) || h->rsplit == 0; }

caar::KernelArgs make_args(const caar_handle_s* h, const caar_control* ctl, double* const* ptr = nullptr) {
  caar::KernelArgs a;
  std::memset(&a, 0, sizeof a);
  if (!ptr) ptr = h->dev;
  a.D = ptr[0]; a.Dinv = ptr[1]; a.fcor = ptr[2]; a.spheremp = ptr[3];
  a.metdet = ptr[4]; a.rmetdet = ptr[5]; a.dp3d = ptr[6]; a.v = ptr[7];
  a.T = ptr[8]; a.phis = ptr[9]; a.Qdp = ptr[10]; a.eta_dot_dpdn = ptr[11];
  a.omega_p = ptr[12]; a.phi = ptr[13]; a.pecnd = ptr[14]; a.vn0 = ptr[15];
  a.nelem = h->dims.nelem; a.nlev = h->dims.nlev; a.qsize_d = h->dims.qsize_d; a.ntl = h->dims.ntl;
  if (ctl) {
    a.nets = ctl->nets; a.nete = ctl->nete; a.n0 = ctl->n0; a.np1 = ctl->np1; a.nm1 = ctl->nm1;
    a.qn0 = ctl->qn0; a.dt2 = ctl->dt2;
  }
  a.rrearth = h->c.rrearth; a.eta_ave_w = h->c.eta_ave_w; a.Rwv = h->c.Rwater_vapor; a.Rgas = h->c.Rgas;
  a.kappa = h->c.kappa; a.hyai0 = h->hyai0; a.ps0 = h->ps0;
  for (int i = 0; i < 16; ++i) a.dvv[i] = h->dvv[i];
  a.tma = h->tma;
  a.rsplit = h->rsplit;
  a.hybi = h->hybi_dev;
  a.lapflat_sched = h->lapflat_sched;
  return a;
}

}  // namespace

extern "C" {

const char* caar_last_error(void) { return g_err; }
const char* caar_version(void) { return "caar_b200 0.1 (sm_100a)"; }

size_t caar_field_count(const caar_dims* dims, int f) {
  if (!dims || f < 0 || f >= CAAR_NUM_FIELDS) return 0;
  return field_count(*dims, f);
}

int caar_device_count(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    fail(CAAR_ERR_CUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    return -CAAR_ERR_CUDA;
  }
  return n;
}

int caar_create(caar_handle* out, const caar_dims* dims, int device) {
  if (!out || !dims) return fail(CAAR_ERR_INVALID, "null argument");
  *out = nullptr;
  if (dims->np != CAAR_NP) return fail(CAAR_ERR_UNSUPPORTED, "np=%d: only np=4 is implemented (reference NP=4)", dims->np);
  if (dims->nelem < 1 || dims->nlev < 2 || dims->qsize_d < 1 || dims->ntl < 1)
    return fail(CAAR_ERR_INVALID, "bad dims nelem=%d nlev=%d qsize_d=%d ntl=%d", dims->nelem, dims->nlev,
                dims->qsize_d, dims->ntl);
  if (caar::strict_smem_bytes(dims->nlev) > 200 * 1024 && !caar::fused_supports(dims->nlev))
    return fail(CAAR_ERR_UNSUPPORTED, "nlev=%d not covered by the compiled kernels", dims->nlev);
  int ndev = 0;
  CU_TRY(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(CAAR_ERR_CUDA, "device %d not available (%d visible)", device, ndev);
  DeviceGuard guard(device);
  if (!guard.ok) return fail(CAAR_ERR_CUDA, "cudaSetDevice(%d) failed", device);
  caar_handle_s* h = new (std::nothrow) caar_handle_s();
  if (!h) return fail(CAAR_ERR_NOMEM, "host allocation failed");
  std::memset(h, 0, sizeof *h);
  h->dims = *dims;
  h->device = device;
  cudaError_t e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreate(&h->ev0);
  if (e == cudaSuccess) e = cudaEventCreate(&h->ev1);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_fence, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->s_in2, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking);
  for (int f = 0; f < CAAR_NUM_FIELDS && e == cudaSuccess; ++f) {
    const size_t bytes = field_count(*dims, f) * sizeof(double);
    e = cudaMalloc(&h->dev[f], bytes);
    if (e == cudaSuccess) e = cudaMemsetAsync(h->dev[f], 0, bytes, h->own_stream);
  }
  if (e == cudaSuccess) e = cudaMalloc(&h->partial, (size_t)dims->nelem * 16 * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&h->bits, (size_t)dims->nelem * 7 * sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaMalloc(&h->out3, 23 * sizeof(double));
  if (e == cudaSuccess) e = cudaMallocHost(&h->out3_host, 23 * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&h->lapflat_sched, 2 * sizeof(unsigned));
  if (e == cudaSuccess) e = cudaMemsetAsync(h->lapflat_sched, 0, 2 * sizeof(unsigned), h->own_stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->own_stream);
  if (e != cudaSuccess) {
    const int code = fail(e == cudaErrorMemoryAllocation ? CAAR_ERR_NOMEM : CAAR_ERR_CUDA, "caar_create: %s",
                          cudaGetErrorString(e));
    char keep[sizeof g_err];
    std::memcpy(keep, g_err, sizeof keep);
    caar_destroy(h);
    std::memcpy(g_err, keep, sizeof keep);
    cudaGetLastError();
    return code;
  }
  h->stream = h->own_stream;
  h->rsplit = 1;
  if (caar::fused_supports(dims->nlev)) {
    h->tma = new (std::nothrow) caar::TmaMaps();
    char msg[256] = "host allocation failed";
    if (!h->tma || caar::build_tma_maps(h->tma, make_args(h, nullptr), msg, sizeof msg)) {
      caar_destroy(h);
      return fail(CAAR_ERR_CUDA, "caar_create: %s", msg);
    }
  }
  *out = h;
  return CAAR_OK;
}

int caar_destroy(caar_handle h) {
  if (!h) return CAAR_OK;
  DeviceGuard guard(h->device);
  if (h->own_stream) cudaStreamSynchronize(h->own_stream);
  for (int f = 0; f < CAAR_NUM_FIELDS; ++f)
    if (h->dev[f]) cudaFree(h->dev[f]);
  if (h->partial) cudaFree(h->partial);
  if (h->bits) cudaFree(h->bits);
  if (h->out3) cudaFree(h->out3);
  if (h->stage) cudaFree(h->stage);
  for (int x = 0; x < CAAR_NUM_EXTRA; ++x)
    if (h->extra[x]) cudaFree(h->extra[x]);
  if (h->hybi_dev) cudaFree(h->hybi_dev);
  if (h->out3_host) cudaFreeHost(h->out3_host);
  if (h->lapflat_sched) cudaFree(h->lapflat_sched);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->ev_fence) cudaEventDestroy(h->ev_fence);
  for (int i = 0; i < h->n_chunk_ev; ++i) cudaEventDestroy(h->chunk_ev[i]);
  delete[] h->chunk_ev;
  if (h->s_in) cudaStreamSynchronize(h->s_in), cudaStreamDestroy(h->s_in);
  if (h->s_in2) cudaStreamSynchronize(h->s_in2), cudaStreamDestroy(h->s_in2);
  if (h->s_out) cudaStreamSynchronize(h->s_out), cudaStreamDestroy(h->s_out);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h->tma;
  delete h->tma_host;
  delete h;
  return CAAR_OK;
}

int caar_set_params(caar_handle h, const caar_constants* c, const double dvv[16], double ps0, const double* hyai) {
  if (!h || !c || !dvv || !hyai) return fail(CAAR_ERR_INVALID, "null argument");
  h->c = *c;
  std::memcpy(h->dvv, dvv, sizeof h->dvv);
  h->ps0 = ps0;
  h->hyai0 = hyai[0];
  h->params_set = true;
  return CAAR_OK;
}

int caar_set_vertical_coordinate(caar_handle h, int rsplit, const double* hybi) {
  if (!h) return fail(CAAR_ERR_INVALID, "null handle");
  if (rsplit < 0) return fail(CAAR_ERR_INVALID, "rsplit=%d", rsplit);
  if (rsplit == 0) {
    if (!hybi) return fail(CAAR_ERR_INVALID, "rsplit=0 (Eulerian) needs hybi[nlev+1]");
    DeviceGuard guard(h->device);
    const size_t bytes = (size_t)(h->dims.nlev + 1) * sizeof(double);
    if (!h->hybi_dev) CU_TRY(cudaMalloc(&h->hybi_dev, bytes));
    CU_TRY(cudaMemcpyAsync(h->hybi_dev, hybi, bytes, cudaMemcpyHostToDevice, h->stream));
    CU_TRY(cudaStreamSynchronize(h->stream));
  }
  h->rsplit = rsplit;
  return CAAR_OK;
}

int caar_set_stream(caar_handle h, void* cuda_stream) {
  if (!h) return fail(CAAR_ERR_INVALID, "null handle");
  cudaStream_t next = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : h->own_stream;
  if (next != h->stream) {  // work already queued on the old stream stays ordered before whatever follows on the new one
    DeviceGuard guard(h->device);
    CU_TRY(cudaEventRecord(h->ev_fence, h->stream));
    CU_TRY(cudaStreamWaitEvent(next, h->ev_fence, 0));
  }
  h->stream = next;
  return CAAR_OK;
}

static int copy_fields(caar_handle h, const caar_arrays* host, unsigned mask, bool to_device) {
  if (!h || !host) return fail(CAAR_ERR_INVALID, "null argument");
  DeviceGuard guard(h->device);
  double* const* tab = as_table(host);
  for (int f = 0; f < CAAR_NUM_FIELDS; ++f) {
    if (!(mask & (1u << f))) continue;
    if (!tab[f]) return fail(CAAR_ERR_INVALID, "host pointer of field %d is null", f);
    const size_t bytes = field_count(h->dims, f) * sizeof(double);
    if (to_device)
      CU_TRY(cudaMemcpyAsync(h->dev[f], tab[f], bytes, cudaMemcpyHostToDevice, h->stream));
    else
      CU_TRY(cudaMemcpyAsync(tab[f], h->dev[f], bytes, cudaMemcpyDeviceToHost, h->stream));
  }
  CU_TRY(cudaStreamSynchronize(h->stream));
  return CAAR_OK;
}

// element range [e0,e1) of the selected fields <-> host arrays that hold ONLY that range
static int copy_range(caar_handle h, const caar_arrays* host, unsigned mask, int e0, int e1, bool to_device) {
  if (!h || !host) return fail(CAAR_ERR_INVALID, "null argument");
  if (e0 < 0 || e1 > h->dims.nelem || e0 > e1) return fail(CAAR_ERR_INVALID, "element range [%d,%d) outside [0,%d)", e0, e1, h->dims.nelem);
  DeviceGuard guard(h->device);
  double* const* tab = as_table(host);
  for (int f = 0; f < CAAR_NUM_FIELDS; ++f) {
    if (!(mask & (1u << f))) continue;
    if (!tab[f]) return fail(CAAR_ERR_INVALID, "host pointer of field %d is null", f);
    const size_t per_elem = field_count(h->dims, f) / h->dims.nelem;
    const size_t bytes = per_elem * (size_t)(e1 - e0) * sizeof(double);
    double* dev = h->dev[f] + per_elem * (size_t)e0;
    if (to_device) CU_TRY(cudaMemcpyAsync(dev, tab[f], bytes, cudaMemcpyHostToDevice, h->stream));
    else CU_TRY(cudaMemcpyAsync(tab[f], dev, bytes, cudaMemcpyDeviceToHost, h->stream));
  }
  CU_TRY(cudaStreamSynchronize(h->stream));
  return CAAR_OK;
}

int caar_upload_range(caar_handle h, const caar_arrays* host, unsigned mask, int e0, int e1) {
  return copy_range(h, host, mask, e0, e1, true);
}
int caar_download_range(caar_handle h, const caar_arrays* host, unsigned mask, int e0, int e1) {
  return copy_range(h, host, mask, e0, e1, false);
}

int caar_upload(caar_handle h, const caar_arrays* host, unsigned mask) { return copy_fields(h, host, mask, true); }
int caar_download(caar_handle h, const caar_arrays* host, unsigned mask) { return copy_fields(h, host, mask, false); }

// ---- Fortran (F90 flat pointer) host layout: copies go through a device staging buffer and a relayout kernel
static const size_t kStageBytes = (size_t)256 << 20;

// block kind of a field for the relayout kernel: 0 = 4x4 scalars, 1 = (u,v) per level, 2 = 2x2 tensors
static int field_kind(int f) { return (f == 0 || f == 1) ? 2 : (f == 7 || f == 15) ? 1 : 0; }

static int copy_fields_f90(caar_handle h, const caar_arrays* host, unsigned mask, bool to_device) {
  if (!h || !host) return fail(CAAR_ERR_INVALID, "null argument");
  DeviceGuard guard(h->device);
  double* const* tab = as_table(host);
  const caar_dims& d = h->dims;
  if (!h->stage) CU_TRY(cudaMalloc(&h->stage, kStageBytes));
  for (int f = 0; f < CAAR_NUM_FIELDS; ++f) {
    if (!(mask & (1u << f))) continue;
    const size_t per_elem = field_count(d, f) / d.nelem;  // doubles
    if (f == 5 && !tab[f] && to_device) {  // HOMMEXX passes no rmetdet (LV/Elements.hpp:92): rmetdet = 1/metdet
      if (!(mask & CAAR_F_METDET) || !tab[4])
        return fail(CAAR_ERR_INVALID, "rmetdet is null: metdet must be uploaded in the same call");
      continue;  // filled after the loop
    }
    if (!tab[f]) return fail(CAAR_ERR_INVALID, "host pointer of field %d is null", f);
    const int kind = field_kind(f);
    const size_t blocks_per_elem = per_elem / (16u << kind);
    size_t chunk = kStageBytes / (per_elem * sizeof(double));
    if (chunk < 1) return fail(CAAR_ERR_UNSUPPORTED, "field %d: one element exceeds the staging buffer", f);
    const int q_dim = (f == 10) ? d.qsize_d : 1;
    for (size_t e0 = 0; e0 < (size_t)d.nelem; e0 += chunk) {
      const size_t ne = ((size_t)d.nelem - e0 < chunk) ? (size_t)d.nelem - e0 : chunk;
      const size_t bytes = ne * per_elem * sizeof(double);
      double* dev = h->dev[f] + e0 * per_elem;
      double* hst = tab[f] + e0 * per_elem;
      if (to_device) {
        CU_TRY(cudaMemcpyAsync(h->stage, hst, bytes, cudaMemcpyHostToDevice, h->stream));
        CU_TRY(caar::launch_relayout(dev, h->stage, ne * blocks_per_elem, kind, true, q_dim, d.nlev,
                                     e0 * blocks_per_elem, h->stream));
      } else {
        CU_TRY(caar::launch_relayout(dev, h->stage, ne * blocks_per_elem, kind, false, q_dim, d.nlev,
                                     e0 * blocks_per_elem, h->stream));
        CU_TRY(cudaMemcpyAsync(hst, h->stage, bytes, cudaMemcpyDeviceToHost, h->stream));
      }
      ++h->launches;
    }
  }
  if (to_device && (mask & CAAR_F_RMETDET) && !tab[5]) {
    CU_TRY(caar::launch_reciprocal(h->dev[5], h->dev[4], field_count(d, 5), h->stream));
    ++h->launches;
  }
  CU_TRY(cudaStreamSynchronize(h->stream));
  return CAAR_OK;
}

int caar_upload_layout(caar_handle h, const caar_arrays* host, unsigned mask, int layout) {
  if (layout == CAAR_LAYOUT_CXX) return copy_fields(h, host, mask, true);
  if (layout == CAAR_LAYOUT_F90) return copy_fields_f90(h, host, mask, true);
  return fail(CAAR_ERR_INVALID, "layout=%d", layout);
}

int caar_download_layout(caar_handle h, const caar_arrays* host, unsigned mask, int layout) {
  if (layout == CAAR_LAYOUT_CXX) return copy_fields(h, host, mask, false);
  if (layout == CAAR_LAYOUT_F90) return copy_fields_f90(h, host, mask, false);
  return fail(CAAR_ERR_INVALID, "layout=%d", layout);
}

int caar_set_params_f90(caar_handle h, const caar_constants* c, const double dvv_f90[16], double ps0,
                        const double* hyai) {
  if (!dvv_f90) return fail(CAAR_ERR_INVALID, "null argument");
  double dvv[16];  // Fortran Dvv(i,j) is stored j-major; the C++ side indexes Dvv[i][j] (F/main.F90:94)
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) dvv[i * 4 + j] = dvv_f90[j * 4 + i];
  return caar_set_params(h, c, dvv, ps0, hyai);
}

int caar_host_register(void* ptr, size_t bytes) {
  if (!ptr || !bytes) return fail(CAAR_ERR_INVALID, "null argument");
  CU_TRY(cudaHostRegister(ptr, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped));
  return CAAR_OK;
}

int caar_host_unregister(void* ptr) {
  if (!ptr) return fail(CAAR_ERR_INVALID, "null argument");
  CU_TRY(cudaHostUnregister(ptr));
  return CAAR_OK;
}

int caar_device_arrays(caar_handle h, caar_arrays* out) {
  if (!h || !out) return fail(CAAR_ERR_INVALID, "null argument");
  std::memcpy(out, h->dev, sizeof h->dev);
  return CAAR_OK;
}

int caar_describe(caar_handle h, int mode, char* buf, size_t len, int* is_fused) {
  if (!h || !buf || !len) return fail(CAAR_ERR_INVALID, "null argument");
  if (mode != CAAR_MODE_FAST && mode != CAAR_MODE_STRICT) return fail(CAAR_ERR_INVALID, "mode=%d", mode);
  const int nlev = h->dims.nlev;
  const bool fused = mode == CAAR_MODE_FAST && caar::fused_supports(nlev);
  if (fused)
    snprintf(buf, len, "caar_fused_kernel<%d,%d,%d>: nlev=%d%s, %d CTA(s) of %d threads per element",
             caar::fused_instance_levels(nlev), caar::fused_instance_cluster(nlev), h->rsplit == 0 ? 1 : 0, nlev,
             caar::fused_instance_levels(nlev) != nlev ? " (padded)" : "", caar::fused_instance_cluster(nlev),
             4 * caar::fused_instance_levels(nlev) / caar::fused_instance_cluster(nlev));
  else
    snprintf(buf, len, "caar_strict_kernel: nlev=%d, one 512-thread CTA per element%s", nlev,
             mode == CAAR_MODE_FAST ? " (FALLBACK: no fused instance for this nlev)" : "");
  if (is_fused) *is_fused = fused ? 1 : 0;
  return CAAR_OK;
}

namespace {

// The checks of caar_run and caar_run_rk5; *fast = the kernel `mode` selects on this handle (fused or strict)
int check_run(caar_handle h, const caar_control* ctl, int nsteps, int mode, const char* who, bool* fast) {
  if (!h) return fail(CAAR_ERR_INVALID, "null handle");
  if (!h->params_set) return fail(CAAR_ERR_STATE, "caar_set_params must be called before %s", who);
  if (int rc = validate_control(h, ctl)) return rc;
  if (nsteps < 0) return fail(CAAR_ERR_INVALID, "nsteps=%d", nsteps);
  if (mode != CAAR_MODE_FAST && mode != CAAR_MODE_STRICT) return fail(CAAR_ERR_INVALID, "mode=%d", mode);
  *fast = uses_fused(h, mode);
  if (!*fast && caar::strict_smem_bytes(h->dims.nlev) > 200 * 1024)
    return fail(CAAR_ERR_UNSUPPORTED, "nlev=%d too large for the strict kernel", h->dims.nlev);
  return CAAR_OK;
}

// ncalls evaluations of compute_and_apply_rhs with the arguments `a` on the handle's stream (caller holds the device)
int launch_rhs(caar_handle h, const caar::KernelArgs& a, int ncalls, bool fast) {
  if (a.nete == a.nets) return CAAR_OK;
  for (int s = 0; s < ncalls; ++s) {
    CU_TRY(fast ? caar::launch_fused(a, h->stream) : caar::launch_strict(a, h->stream));
    ++h->launches;
  }
  return CAAR_OK;
}

}  // namespace

int caar_run(caar_handle h, const caar_control* ctl, int nsteps, int mode) {
  bool fast = false;
  if (int rc = check_run(h, ctl, nsteps, mode, "caar_run", &fast)) return rc;
  DeviceGuard guard(h->device);
  return launch_rhs(h, make_args(h, ctl), nsteps, fast);
}

int caar_run_rk5(caar_handle h, caar_control* ctl, double dt, int nsteps, int mode) {
  bool fast = false;
  if (int rc = check_run(h, ctl, nsteps, mode, "caar_run_rk5", &fast)) return rc;
  if (ctl->n0 == ctl->np1 || ctl->n0 == ctl->nm1 || ctl->np1 == ctl->nm1)  // stage 1 would overwrite u0
    return fail(CAAR_ERR_INVALID, "caar_run_rk5 needs pairwise distinct time levels (n0=%d np1=%d nm1=%d)", ctl->n0,
                ctl->np1, ctl->nm1);
  DeviceGuard guard(h->device);
  const double w = h->c.eta_ave_w;
  for (int s = 0; s < nsteps; ++s) {
    const int n0 = ctl->n0, np1 = ctl->np1, nm1 = ctl->nm1;
    // prim_advance_exp, tstep_type == 5: {n0, np1, nm1, dt2, eta_ave_w} of the five compute_and_apply_rhs calls
    const struct { int n0, np1, nm1; double dt2, eta_ave_w; } stage[5] = {
        {n0, nm1, n0, dt / 5, w / 4},          {nm1, np1, n0, dt / 5, 0.0},          {np1, np1, n0, dt / 3, 0.0},
        {np1, np1, n0, (2 * dt) / 3, 0.0},     {np1, np1, nm1, (3 * dt) / 4, (3 * w) / 4}};
    for (int k = 0; k < 5 && ctl->nete > ctl->nets; ++k) {
      if (k == 4) {  // u(nm1) = (5 u1 - u0)/4
        CU_TRY(caar::launch_rk5_combine(make_args(h, ctl), ctl->nets, ctl->nete, nm1, n0, h->stream));
        ++h->launches;
      }
      caar::KernelArgs a = make_args(h, ctl);
      a.n0 = stage[k].n0;
      a.np1 = stage[k].np1;
      a.nm1 = stage[k].nm1;
      a.dt2 = stage[k].dt2;
      a.eta_ave_w = stage[k].eta_ave_w;
      if (int rc = launch_rhs(h, a, 1, fast)) return rc;
    }
    caar_update_time_levels(ctl);
  }
  return CAAR_OK;
}

// ---- caar_run_host: one RHS evaluation on HOST arrays, pipelined over element chunks --------------------
namespace {

// one contiguous run of doubles inside every element's block of a field
struct Slice {
  int f;            // field index (order of caar_arrays)
  size_t per_elem;  // doubles per element of the whole field
  size_t off, len;  // the run [off, off+len) inside the element's block
};

// true when every host array is page-locked and mapped into the device address space; dev[] = device aliases
bool host_arrays_mapped(double* const* tab, double** dev) {
  for (int f = 0; f < CAAR_NUM_FIELDS; ++f) {
    dev[f] = nullptr;
    if (!tab[f]) return false;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, tab[f]) != cudaSuccess) {
      cudaGetLastError();
      return false;
    }
    if (at.type != cudaMemoryTypeHost || !at.devicePointer) return false;
    dev[f] = static_cast<double*>(at.devicePointer);
  }
  return true;
}

bool zero_copy_default() {
  static const int v = [] {
    const char* e = getenv("CAAR_HOST_PATH");  // "staged" | "zerocopy"
    if (e && std::strcmp(e, "staged") == 0) return 0;
    if (e && std::strcmp(e, "zerocopy") == 0) return 1;
    return CAAR_HOST_DEFAULT_ZERO_COPY;
  }();
  return v != 0;
}

int add_levels(Slice* out, int n, int f, size_t lf, int ntl, int tl_a, int tl_b) {
  out[n++] = Slice{f, lf * ntl, lf * tl_a, lf};
  if (tl_b != tl_a) out[n++] = Slice{f, lf * ntl, lf * tl_b, lf};
  return n;
}

cudaError_t copy_slice(const Slice& s, double* dev, double* host, int e0, int e1, bool to_device, cudaStream_t st) {
  const size_t n = (size_t)(e1 - e0);
  double* d = dev + (size_t)e0 * s.per_elem + s.off;
  double* h = host + (size_t)e0 * s.per_elem + s.off;
  const cudaMemcpyKind kind = to_device ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost;
  if (s.len == s.per_elem)
    return to_device ? cudaMemcpyAsync(d, h, n * s.len * sizeof(double), kind, st)
                     : cudaMemcpyAsync(h, d, n * s.len * sizeof(double), kind, st);
  const size_t pitch = s.per_elem * sizeof(double), width = s.len * sizeof(double);
  // Pitched DMA over PCIe runs markedly slower with 18 KB rows than with 9 KB rows while the other direction
  // is busy (measured: tools/pcie_probe.cu, profiles/README.md), so wide rows are cut into pieces of <= row_max B
  static const size_t row_max = [] { const char* e = getenv("CAAR_HOST_ROW"); return e ? (size_t)atol(e) : (size_t)9216; }();
  static const int split_dirs = [] { const char* e = getenv("CAAR_HOST_SPLIT"); return e ? atoi(e) : 3; }();  // 1 = in, 2 = out
  if (row_max > 0 && width > row_max && (split_dirs & (to_device ? 1 : 2))) {
    for (size_t o = 0; o < width; o += row_max) {
      const size_t wd = (width - o < row_max) ? width - o : row_max;
      const cudaError_t e = to_device ? cudaMemcpy2DAsync((char*)d + o, pitch, (char*)h + o, pitch, wd, n, kind, st)
                                      : cudaMemcpy2DAsync((char*)h + o, pitch, (char*)d + o, pitch, wd, n, kind, st);
      if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
  }
  return to_device ? cudaMemcpy2DAsync(d, pitch, h, pitch, width, n, kind, st)
                   : cudaMemcpy2DAsync(h, pitch, d, pitch, width, n, kind, st);
}

}  // namespace

int caar_run_host(caar_handle h, const caar_arrays* host, const caar_control* ctl, int mode, int chunk_elems) {
  if (!h || !host) return fail(CAAR_ERR_INVALID, "null argument");
  if (!h->params_set) return fail(CAAR_ERR_STATE, "caar_set_params must be called before caar_run_host");
  if (int rc = validate_control(h, ctl)) return rc;
  if (mode != CAAR_MODE_FAST && mode != CAAR_MODE_STRICT) return fail(CAAR_ERR_INVALID, "mode=%d", mode);
  if (chunk_elems < 0 && chunk_elems != CAAR_HOST_ZERO_COPY) return fail(CAAR_ERR_INVALID, "chunk_elems=%d", chunk_elems);
  const caar_dims& d = h->dims;
  const bool fast = uses_fused(h, mode);
  if (!fast && caar::strict_smem_bytes(d.nlev) > 200 * 1024)
    return fail(CAAR_ERR_UNSUPPORTED, "nlev=%d too large for the strict kernel", d.nlev);
  const int n = ctl->nete - ctl->nets;
  if (n == 0) return CAAR_OK;

  // the slices the routine reads (PO/compute_and_apply_rhs.cpp:74-257) and writes (:117,161,172-173,251-254)
  const size_t lf = (size_t)d.nlev * 16;
  Slice in[24], out[8];
  int ni = 0, no = 0;
  for (int f : {0, 1, 2, 3, 4, 5, 9}) in[ni++] = Slice{f, field_count(d, f) / d.nelem, 0, field_count(d, f) / d.nelem};
  ni = add_levels(in, ni, 6, lf, d.ntl, ctl->n0, ctl->nm1);
  ni = add_levels(in, ni, 7, 2 * lf, d.ntl, ctl->n0, ctl->nm1);
  ni = add_levels(in, ni, 8, lf, d.ntl, ctl->n0, ctl->nm1);
  if (ctl->qn0 != -1) in[ni++] = Slice{10, lf * 2 * d.qsize_d, lf * ctl->qn0, lf};
  in[ni++] = Slice{12, lf, 0, lf};
  in[ni++] = Slice{14, lf, 0, lf};
  in[ni++] = Slice{15, 2 * lf, 0, 2 * lf};
  out[no++] = Slice{6, lf * d.ntl, lf * ctl->np1, lf};
  out[no++] = Slice{7, 2 * lf * d.ntl, 2 * lf * ctl->np1, 2 * lf};
  out[no++] = Slice{8, lf * d.ntl, lf * ctl->np1, lf};
  out[no++] = Slice{12, lf, 0, lf};
  out[no++] = Slice{13, lf, 0, lf};
  out[no++] = Slice{15, 2 * lf, 0, 2 * lf};
  if (moves_eta(h, mode)) {  // reference-order kernel: eta_dot_dpdn += eta_ave_w*0 (PO:164-171); Eulerian: the real flux
    const size_t le = (size_t)(d.nlev + 1) * 16;
    in[ni++] = Slice{11, le, 0, le};
    out[no++] = Slice{11, le, 0, le};
  }
  double* const* tab = as_table(host);
  for (int i = 0; i < ni; ++i)
    if (!tab[in[i].f]) return fail(CAAR_ERR_INVALID, "host pointer of field %d is null", in[i].f);
  for (int i = 0; i < no; ++i)
    if (!tab[out[i].f]) return fail(CAAR_ERR_INVALID, "host pointer of field %d is null", out[i].f);

  DeviceGuard guard(h->device);
  // ---- zero-copy path: the kernel itself reads the caller's arrays over PCIe (TMA / LDG on mapped host memory)
  // and writes the results straight back: one launch, both link directions busy, no staging copies
  double* mapped[CAAR_NUM_FIELDS];
  const bool can_map = host_arrays_mapped(tab, mapped);
  if (chunk_elems == CAAR_HOST_ZERO_COPY && !can_map)
    return fail(CAAR_ERR_INVALID, "CAAR_HOST_ZERO_COPY needs page-locked, device-mapped host arrays "
                                  "(caar_host_register / cudaHostAlloc)");
  if (can_map && (chunk_elems == CAAR_HOST_ZERO_COPY || (chunk_elems == 0 && zero_copy_default()))) {
    caar::KernelArgs za = make_args(h, ctl, mapped);
    za.tma = nullptr;
    za.pf_dist = -1;  // no L2 prefetch of host memory
    if (caar::fused_supports(d.nlev)) {
      if (!h->tma_host || std::memcmp(h->tma_host_key, mapped, sizeof mapped) != 0) {
        if (!h->tma_host) h->tma_host = new (std::nothrow) caar::TmaMaps();
        char msg[256] = "host allocation failed";
        if (!h->tma_host || caar::build_tma_maps(h->tma_host, za, msg, sizeof msg)) {
          delete h->tma_host;
          h->tma_host = nullptr;
          return fail(CAAR_ERR_CUDA, "caar_run_host: %s", msg);
        }
        std::memcpy(h->tma_host_key, mapped, sizeof mapped);
      }
      za.tma = h->tma_host;
    }
    CU_TRY(fast ? caar::launch_fused(za, h->stream) : caar::launch_strict(za, h->stream));
    ++h->launches;
    CU_TRY(cudaStreamSynchronize(h->stream));
    return CAAR_OK;
  }

  // ---- staged path. Chunking: enough chunks to hide the first copy-in and the last copy-out, big enough to keep
  // every SM busy
  int chunk = chunk_elems;
  if (chunk == 0) {
    chunk = (n + 47) / 48;
    if (chunk < 296) chunk = 296;
    if (chunk > 4096) chunk = 4096;
  }
  // After the last copy-in nothing overlaps the last kernel and copy-out: the tail of the range is cut finer (the last
  // chunk in halves, three times), which shortens that drain from one chunk's copy-out to an eighth of it
  const int full = (n + chunk - 1) / chunk;
  int tail[5] = {ctl->nets + (full - 1) * chunk, ctl->nete, 0, 0, 0}, ntail = 1;  // boundaries of the pieces of the last chunk
  for (int k = 0; k < 3 && chunk_elems == 0; ++k) {
    const int a0 = tail[ntail - 1], a1 = tail[ntail];
    if (a1 - a0 < 2 * 296) break;
    tail[ntail] = a0 + (a1 - a0) / 2;
    tail[++ntail] = a1;
  }
  const int nchunks = full - 1 + ntail;
  if (h->n_chunk_ev < 3 * nchunks) {
    cudaEvent_t* ev = new (std::nothrow) cudaEvent_t[3 * nchunks];
    if (!ev) return fail(CAAR_ERR_NOMEM, "host allocation failed");
    for (int i = 0; i < h->n_chunk_ev; ++i) ev[i] = h->chunk_ev[i];
    delete[] h->chunk_ev;
    h->chunk_ev = ev;
    while (h->n_chunk_ev < 3 * nchunks) {
      CU_TRY(cudaEventCreateWithFlags(&h->chunk_ev[h->n_chunk_ev], cudaEventDisableTiming));
      ++h->n_chunk_ev;
    }
  }
  // the copy-in stream must not overtake work already queued on the compute stream (it rewrites the mirrors)
  CU_TRY(cudaEventRecord(h->ev_fence, h->stream));
  CU_TRY(cudaStreamWaitEvent(h->s_in, h->ev_fence, 0));
  // the copy-in of a chunk may be dealt over two streams (two copy engines reading the host at once)
  static const int in_streams = [] { const char* e = getenv("CAAR_HOST_IN_STREAMS"); return e ? atoi(e) : 1; }();
  if (in_streams > 1) CU_TRY(cudaStreamWaitEvent(h->s_in2, h->ev_fence, 0));
  caar::KernelArgs a = make_args(h, ctl);
  // On any failure inside the pipeline the three streams are drained before returning, so that no DMA is still
  // reading or writing the caller's arrays when the caller sees the error (the host arrays may then hold the results
  // of the chunks that completed: the call is NOT transactional).
  cudaError_t ce = cudaSuccess;
  const char* what = "";
#define PIPE_TRY(expr)            \
  if (ce == cudaSuccess) {        \
    ce = (expr);                  \
    if (ce != cudaSuccess) what = #expr; \
  }
  for (int c = 0; c < nchunks && ce == cudaSuccess; ++c) {
    const int e0 = c < full - 1 ? ctl->nets + c * chunk : tail[c - (full - 1)];
    const int e1 = c < full - 1 ? e0 + chunk : tail[c - (full - 1) + 1];
    for (int i = 0; i < ni; ++i)
      PIPE_TRY(copy_slice(in[i], h->dev[in[i].f], tab[in[i].f], e0, e1, true, (in_streams > 1 && (i & 1)) ? h->s_in2 : h->s_in));
    PIPE_TRY(cudaEventRecord(h->chunk_ev[2 * c], h->s_in));
    PIPE_TRY(cudaStreamWaitEvent(h->stream, h->chunk_ev[2 * c], 0));
    if (in_streams > 1) {
      PIPE_TRY(cudaEventRecord(h->chunk_ev[2 * nchunks + c], h->s_in2));
      PIPE_TRY(cudaStreamWaitEvent(h->stream, h->chunk_ev[2 * nchunks + c], 0));
    }
    a.nets = e0;
    a.nete = e1;
    PIPE_TRY(fast ? caar::launch_fused(a, h->stream) : caar::launch_strict(a, h->stream));
    if (ce == cudaSuccess) ++h->launches;
    PIPE_TRY(cudaEventRecord(h->chunk_ev[2 * c + 1], h->stream));
    PIPE_TRY(cudaStreamWaitEvent(h->s_out, h->chunk_ev[2 * c + 1], 0));
    for (int i = 0; i < no; ++i) PIPE_TRY(copy_slice(out[i], h->dev[out[i].f], tab[out[i].f], e0, e1, false, h->s_out));
  }
#undef PIPE_TRY
  if (ce != cudaSuccess) {
    cudaStreamSynchronize(h->s_in);
    cudaStreamSynchronize(h->s_in2);
    cudaStreamSynchronize(h->stream);
    cudaStreamSynchronize(h->s_out);
    cudaGetLastError();
    return fail(ce == cudaErrorMemoryAllocation ? CAAR_ERR_NOMEM : CAAR_ERR_CUDA, "caar_run_host: %s failed: %s", what,
                cudaGetErrorString(ce));
  }
  CU_TRY(cudaStreamSynchronize(h->s_out));
  CU_TRY(cudaStreamSynchronize(h->stream));
  return CAAR_OK;
}

int caar_host_traffic(caar_handle h, const caar_control* ctl, int mode, size_t* h2d_bytes, size_t* d2h_bytes) {
  if (!h || !ctl || !h2d_bytes || !d2h_bytes) return fail(CAAR_ERR_INVALID, "null argument");
  if (int rc = validate_control(h, ctl)) return rc;
  const caar_dims& d = h->dims;
  const bool fast = uses_fused(h, mode);
  const size_t lf = (size_t)d.nlev * 16, le = (size_t)(d.nlev + 1) * 16;
  const size_t lv = (ctl->n0 == ctl->nm1) ? 1 : 2;
  (void)fast;
  const size_t eta = moves_eta(h, mode) ? le : 0;
  size_t in = 2 * 64 + 5 * 16 + lv * 4 * lf + (ctl->qn0 != -1 ? lf : 0) + 4 * lf + eta;
  size_t out = 8 * lf + eta;
  const size_t n = (size_t)(ctl->nete - ctl->nets);
  *h2d_bytes = in * n * sizeof(double);
  *d2h_bytes = out * n * sizeof(double);
  return CAAR_OK;
}

// ---- tracer step after CAAR ---------------------------------------------------------------------------------
size_t caar_extra_count(const caar_dims* d, int which) {
  if (!d) return 0;
  if (which == CAAR_X_VSTAR) return (size_t)d->nelem * d->nlev * 32;
  if (which == CAAR_X_QTENS) return (size_t)d->nelem * d->qsize_d * d->nlev * 16;
  if (which == CAAR_X_TENSORVISC) return (size_t)d->nelem * 64;
  if (which == CAAR_X_SCALAR_IN || which == CAAR_X_SCALAR_OUT) return (size_t)d->nelem * d->nlev * 16;
  return 0;
}

static int extra_buffer(caar_handle h, int which, double** out) {
  if (!h) return fail(CAAR_ERR_INVALID, "null handle");
  if (which < 0 || which >= CAAR_NUM_EXTRA) return fail(CAAR_ERR_INVALID, "extra array %d", which);
  if (!h->extra[which]) {
    const size_t bytes = caar_extra_count(&h->dims, which) * sizeof(double);
    CU_TRY(cudaMalloc(&h->extra[which], bytes));
    CU_TRY(cudaMemsetAsync(h->extra[which], 0, bytes, h->stream));
  }
  *out = h->extra[which];
  return CAAR_OK;
}

int caar_extra_upload(caar_handle h, int which, const double* host) {
  if (!host) return fail(CAAR_ERR_INVALID, "null argument");
  double* dev = nullptr;
  if (!h) return fail(CAAR_ERR_INVALID, "null handle");
  DeviceGuard guard(h->device);
  if (int rc = extra_buffer(h, which, &dev)) return rc;
  CU_TRY(cudaMemcpyAsync(dev, host, caar_extra_count(&h->dims, which) * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  CU_TRY(cudaStreamSynchronize(h->stream));
  return CAAR_OK;
}

int caar_extra_download(caar_handle h, int which, double* host) {
  if (!host) return fail(CAAR_ERR_INVALID, "null argument");
  double* dev = nullptr;
  if (!h) return fail(CAAR_ERR_INVALID, "null handle");
  DeviceGuard guard(h->device);
  if (int rc = extra_buffer(h, which, &dev)) return rc;
  CU_TRY(cudaMemcpyAsync(host, dev, caar_extra_count(&h->dims, which) * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(cudaStreamSynchronize(h->stream));
  return CAAR_OK;
}

namespace {

// The checks of caar_euler_step and caar_advect_tracers
int check_euler(caar_handle h, int nets, int nete, int qn0, int qsize, int mode, const char* who) {
  if (!h) return fail(CAAR_ERR_INVALID, "null handle");
  if (!h->params_set) return fail(CAAR_ERR_STATE, "caar_set_params must be called before %s", who);
  if (nets < 0 || nete > h->dims.nelem || nets > nete) return fail(CAAR_ERR_INVALID, "element range [%d,%d)", nets, nete);
  if (qn0 < 0 || qn0 > 1) return fail(CAAR_ERR_INVALID, "qn0=%d must be 0 or 1", qn0);
  if (qsize < 0 || qsize > h->dims.qsize_d) return fail(CAAR_ERR_INVALID, "qsize=%d outside [0,%d]", qsize, h->dims.qsize_d);
  if (mode != CAAR_MODE_FAST && mode != CAAR_MODE_STRICT) return fail(CAAR_ERR_INVALID, "mode=%d", mode);
  return CAAR_OK;
}

// One tracer step Qdp(qn0) - dt div(vstar Qdp(qn0)) on the handle's stream (caller holds the device); tracer iq of
// element e goes to the level slice (e * qsize_d + iq) * out_stride + out_off of `out`: (qtens, 1, 0) or (Qdp, 2, np1).
// Fast mode: the TMA-pipelined level-local skeleton (caar_levelops.cu); CAAR_EULER_V1=1 keeps the first-generation
// LDG/STG kernel for A/B runs. Strict mode: the reference-order kernel of caar_euler.cu.
int launch_tracer_step(caar_handle h, const caar::KernelArgs& a, const double* vstar, double* out, int out_stride,
                       int out_off, int nets, int nete, int qn0, int qsize, double dt, int mode) {
  static const bool v1 = [] { const char* e = getenv("CAAR_EULER_V1"); return e && atoi(e) != 0; }();
  if (mode == CAAR_MODE_STRICT || v1)
    CU_TRY(caar::launch_euler_step(a, vstar, out, out_stride, out_off, nets, nete, qn0, qsize, dt,
                                   mode == CAAR_MODE_STRICT, h->stream));
  else
    CU_TRY(caar::launch_levelop(0, a, a.Qdp, vstar, out, nullptr, nets, nete, qn0, qsize, dt, out_stride, out_off,
                                false, h->stream));
  if (nete > nets && qsize > 0) ++h->launches;
  return CAAR_OK;
}

}  // namespace

int caar_euler_step(caar_handle h, int nets, int nete, int qn0, int qsize, double dt, int mode) {
  if (int rc = check_euler(h, nets, nete, qn0, qsize, mode, "caar_euler_step")) return rc;
  DeviceGuard guard(h->device);
  double *vstar = nullptr, *qtens = nullptr;
  if (int rc = extra_buffer(h, CAAR_X_VSTAR, &vstar)) return rc;
  if (int rc = extra_buffer(h, CAAR_X_QTENS, &qtens)) return rc;
  return launch_tracer_step(h, make_args(h, nullptr), vstar, qtens, 1, 0, nets, nete, qn0, qsize, dt, mode);
}

int caar_advect_tracers(caar_handle h, int nets, int nete, int* qn0, int qsize, double dt, int nsteps, int mode) {
  if (!qn0) return fail(CAAR_ERR_INVALID, "qn0 is null");
  if (int rc = check_euler(h, nets, nete, *qn0, qsize, mode, "caar_advect_tracers")) return rc;
  if (nsteps < 0) return fail(CAAR_ERR_INVALID, "nsteps=%d", nsteps);
  DeviceGuard guard(h->device);
  double* vstar = nullptr;
  if (int rc = extra_buffer(h, CAAR_X_VSTAR, &vstar)) return rc;
  const caar::KernelArgs a = make_args(h, nullptr);
  double* Qdp = const_cast<double*>(a.Qdp);  // the handle's own mirror; const in KernelArgs for the kernels that read it
  const double half = dt / 2;
  for (int s = 0; s < nsteps; ++s) {
    const int n0 = *qn0, np1 = 1 - n0;
    if (nete > nets && qsize > 0) {
      // three euler_step stages of dt/2 into Qdp(np1), stages 2 and 3 in place, then the time average
      for (int k = 0; k < 3; ++k)
        if (int rc = launch_tracer_step(h, a, vstar, Qdp, 2, np1, nets, nete, k == 0 ? n0 : np1, qsize, half, mode))
          return rc;
      CU_TRY(caar::launch_qdp_avg(a, nets, nete, qsize, n0, np1, h->stream));
      ++h->launches;
    }
    *qn0 = np1;  // TimeLevel_Qdp: n0_qdp <-> np1_qdp
  }
  return CAAR_OK;
}

int caar_sphere_wk(caar_handle h, int op, int nets, int nete, int mode) {
  if (!h) return fail(CAAR_ERR_INVALID, "null handle");
  if (!h->params_set) return fail(CAAR_ERR_STATE, "caar_set_params must be called before caar_sphere_wk");
  if (nets < 0 || nete > h->dims.nelem || nets > nete) return fail(CAAR_ERR_INVALID, "element range [%d,%d)", nets, nete);
  if (op < CAAR_OP_DIVERGENCE_WK || op > CAAR_OP_LAPLACE_TENSOR_REPLACE) return fail(CAAR_ERR_INVALID, "op=%d", op);
  if (mode != CAAR_MODE_FAST && mode != CAAR_MODE_STRICT) return fail(CAAR_ERR_INVALID, "mode=%d", mode);
  DeviceGuard guard(h->device);
  double *vin = nullptr, *sin = nullptr, *out = nullptr, *tv = nullptr;
  if (int rc = extra_buffer(h, CAAR_X_SCALAR_OUT, &out)) return rc;
  if (op == CAAR_OP_DIVERGENCE_WK) {
    if (int rc = extra_buffer(h, CAAR_X_VSTAR, &vin)) return rc;
  } else if (op == CAAR_OP_LAPLACE_TENSOR_REPLACE) {
    sin = out;
  } else {
    if (int rc = extra_buffer(h, CAAR_X_SCALAR_IN, &sin)) return rc;
  }
  if (op == CAAR_OP_LAPLACE_TENSOR || op == CAAR_OP_LAPLACE_TENSOR_REPLACE)
    if (int rc = extra_buffer(h, CAAR_X_TENSORVISC, &tv)) return rc;
  const caar::KernelArgs a = make_args(h, nullptr);
  const int kop = op == CAAR_OP_DIVERGENCE_WK ? 1 : op == CAAR_OP_LAPLACE_SIMPLE ? 2 : 3;
  CU_TRY(caar::launch_levelop(kop, a, kop == 1 ? vin : sin, nullptr, out, tv, nets, nete, 0, 1, 0.0, 1, 0,
                              mode == CAAR_MODE_STRICT, h->stream));
  if (nete > nets) ++h->launches;
  return CAAR_OK;
}

void caar_update_time_levels(caar_control* ctl) {
  if (!ctl) return;
  const int tmp = ctl->np1;  // TestData::update_time_levels, PO/data_structures.cpp:174-180
  ctl->np1 = ctl->nm1;
  ctl->nm1 = ctl->n0;
  ctl->n0 = tmp;
}

int caar_run_stepping(caar_handle h, caar_control* ctl, int nsteps, int mode) {
  if (!ctl) return fail(CAAR_ERR_INVALID, "control is null");
  if (nsteps < 0) return fail(CAAR_ERR_INVALID, "nsteps=%d", nsteps);
  for (int s = 0; s < nsteps; ++s) {
    if (int rc = caar_run(h, ctl, 1, mode)) return rc;
    caar_update_time_levels(ctl);
  }
  return CAAR_OK;
}

int caar_sync(caar_handle h) {
  if (!h) return fail(CAAR_ERR_INVALID, "null handle");
  DeviceGuard guard(h->device);
  CU_TRY(cudaStreamSynchronize(h->stream));
  return CAAR_OK;
}

long long caar_launch_count(caar_handle h) { return h ? h->launches : 0; }

int caar_timer_start(caar_handle h) {
  if (!h) return fail(CAAR_ERR_INVALID, "null handle");
  DeviceGuard guard(h->device);
  CU_TRY(cudaEventRecord(h->ev0, h->stream));
  return CAAR_OK;
}

int caar_timer_stop(caar_handle h, float* ms) {
  if (!h || !ms) return fail(CAAR_ERR_INVALID, "null argument");
  DeviceGuard guard(h->device);
  CU_TRY(cudaEventRecord(h->ev1, h->stream));
  CU_TRY(cudaEventSynchronize(h->ev1));
  CU_TRY(cudaEventElapsedTime(ms, h->ev0, h->ev1));
  return CAAR_OK;
}

int caar_norms(caar_handle h, int tl, int nets, int nete, double sumsq[3]) {
  if (!h || !sumsq) return fail(CAAR_ERR_INVALID, "null argument");
  if (tl < 0 || tl >= h->dims.ntl) return fail(CAAR_ERR_INVALID, "time level %d", tl);
  if (nets < 0 || nete > h->dims.nelem || nets > nete) return fail(CAAR_ERR_INVALID, "element range [%d,%d)", nets, nete);
  DeviceGuard guard(h->device);
  const caar::KernelArgs a = make_args(h, nullptr);
  CU_TRY(caar::launch_norms(a, tl, nets, nete, h->partial, h->out3, h->stream));
  h->launches += (nete > nets) ? 2 : 1;
  CU_TRY(cudaMemcpyAsync(h->out3_host, h->out3, 3 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(cudaStreamSynchronize(h->stream));
  for (int i = 0; i < 3; ++i) sumsq[i] = h->out3_host[i];
  return CAAR_OK;
}

int caar_checksums(caar_handle h, int tl, int nets, int nete, caar_checksum* out) {
  if (!h || !out) return fail(CAAR_ERR_INVALID, "null argument");
  if (tl < 0 || tl >= h->dims.ntl) return fail(CAAR_ERR_INVALID, "time level %d", tl);
  if (nets < 0 || nete > h->dims.nelem || nets > nete) return fail(CAAR_ERR_INVALID, "element range [%d,%d)", nets, nete);
  DeviceGuard guard(h->device);
  const caar::KernelArgs a = make_args(h, nullptr);
  unsigned long long* out7 = reinterpret_cast<unsigned long long*>(h->out3 + 16);
  CU_TRY(caar::launch_checksums(a, tl, nets, nete, h->c.cp, h->partial, h->bits, h->out3, out7, h->stream));
  h->launches += (nete > nets) ? 2 : 1;
  CU_TRY(cudaMemcpyAsync(h->out3_host, h->out3, 23 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU_TRY(cudaStreamSynchronize(h->stream));
  for (int f = 0; f < 7; ++f) {
    out->sum[f] = h->out3_host[2 * f];
    out->sumsq[f] = h->out3_host[2 * f + 1];
    std::memcpy(&out->bits[f], &h->out3_host[16 + f], sizeof(unsigned long long));
  }
  out->energy[0] = h->out3_host[14];
  out->energy[1] = h->out3_host[15];
  return CAAR_OK;
}

int caar_compute_and_apply_rhs_host(const caar_dims* dims, const caar_arrays* host, const caar_control* ctl,
                                    const caar_constants* c, const double dvv[16], double ps0,
                                    const double* hyai, int device, int mode) {
  caar_handle h = nullptr;
  int rc = caar_create(&h, dims, device);
  if (rc) return rc;
  rc = caar_set_params(h, c, dvv, ps0, hyai);
  if (!rc) rc = caar_run_host(h, host, ctl, mode, 0);
  char keep[sizeof g_err];
  std::memcpy(keep, g_err, sizeof keep);
  caar_destroy(h);
  std::memcpy(g_err, keep, sizeof keep);
  return rc;
}

int caar_saxpby_device(double a, double b, double* x_dev, const double* y_dev, size_t n, void* cuda_stream) {
  if (!x_dev || !y_dev) return fail(CAAR_ERR_INVALID, "null argument");
  CU_TRY(caar::launch_saxpby(a, b, x_dev, y_dev, n, static_cast<cudaStream_t>(cuda_stream)));
  return CAAR_OK;
}

int caar_saxpby_host(double a, double b, double* x, const double* y, size_t n, int sweeps, int device) {
  if (!x || !y) return fail(CAAR_ERR_INVALID, "null argument");
  int ndev = 0;
  CU_TRY(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(CAAR_ERR_CUDA, "device %d not available", device);
  DeviceGuard guard(device);
  double *dx = nullptr, *dy = nullptr;
  CU_TRY(cudaMalloc(&dx, n * sizeof(double)));
  cudaError_t e = cudaMalloc(&dy, n * sizeof(double));
  if (e == cudaSuccess) e = cudaMemcpy(dx, x, n * sizeof(double), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(dy, y, n * sizeof(double), cudaMemcpyHostToDevice);
  for (int s = 0; s < sweeps && e == cudaSuccess; ++s) e = caar::launch_saxpby(a, b, dx, dy, n, 0);
  if (e == cudaSuccess) e = cudaMemcpy(x, dx, n * sizeof(double), cudaMemcpyDeviceToHost);
  cudaFree(dx);
  cudaFree(dy);
  if (e != cudaSuccess) return fail(CAAR_ERR_CUDA, "caar_saxpby_host: %s", cudaGetErrorString(e));
  return CAAR_OK;
}

}  // extern "C"
