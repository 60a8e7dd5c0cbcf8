// caar_fused.cu — dispatch of CAAR_MODE_FAST to the fused kernel instances (caar_fused_kernel.cuh), the TMA tensor
// maps they use, and the instances for the two level counts of the reference configurations (nlev = 72, 128).
// The other instances (multiples of 8 up to 64, 80, 96, 112, 120) are in caar_fused_more.cu; a level count without
// an instance of its own runs on the next larger one with padding levels (instance_for()).
#include "caar_fused_kernel.cuh"

namespace caar {
int encode_tma_map(CUtensorMap* m, const void* base, cuuint64_t slices, cuuint64_t rows, cuuint32_t box_rows,
                   const char* name, char* err, size_t errlen) {
  typedef CUresult (*encode_t)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                               const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                               CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static cudaError_t lookup = cudaSuccess;
  static const encode_t encode = [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    lookup = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    return lookup == cudaSuccess && fn && qres == cudaDriverEntryPointSuccess ? reinterpret_cast<encode_t>(fn) : nullptr;
  }();
  if (!encode) {
    snprintf(err, errlen, "cuTensorMapEncodeTiled entry point unavailable (%s)", cudaGetErrorString(lookup));
    return 1;
  }
  if (box_rows > 256 || slices >= (1ull << 31)) {
    snprintf(err, errlen, "tensor map %s: box of %u rows / %llu slices out of range", name, box_rows,
             (unsigned long long)slices);
    return 1;
  }
  const cuuint64_t gdim[3] = {16, rows, slices};
  const cuuint64_t gstride[2] = {128, rows * 128};
  const cuuint32_t box[3] = {16, box_rows, 1};
  const cuuint32_t estride[3] = {1, 1, 1};
  const CUresult r = encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, const_cast<void*>(base), gdim, gstride, box, estride,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(err, errlen, "cuTensorMapEncodeTiled(%s) failed with CUresult %d", name, (int)r);
    return 1;
  }
  return 0;
}

int build_tma_maps(TmaMaps* out, const KernelArgs& a, char* err, size_t errlen) {
  const cuuint64_t E = (cuuint64_t)a.nelem, L = (cuuint64_t)a.nlev, ntl = (cuuint64_t)a.ntl;
  const int inst = instance_for(a.nlev);  // compiled level count serving this nlev (>= nlev)
  const cuuint32_t LB = (cuuint32_t)(inst / (cluster_for(inst) > 0 ? cluster_for(inst) : 1));  // levels per CTA = box rows
  // every array as [slices][rows][16 doubles]: rows = the levels of one element (x time level, tracer ...) slice, x2 for
  // the interleaved (u,v) fields. A box that sticks out of its slice (padding levels) costs no HBM traffic.
  struct Spec { CUtensorMap* m; const void* base; cuuint64_t slices; cuuint64_t rows; cuuint32_t box; const char* name; };
  const Spec specs[8] = {
      {&out->Qdp, a.Qdp, E * (cuuint64_t)a.qsize_d * 2, L, LB, "Qdp"},
      {&out->dp3d, a.dp3d, E * ntl, L, LB, "dp3d"},
      {&out->T, a.T, E * ntl, L, LB, "T"},
      {&out->v, a.v, E * ntl, 2 * L, 2 * LB, "v"},
      {&out->vn0, a.vn0, E, 2 * L, 2 * LB, "vn0"},
      {&out->pecnd, a.pecnd, E, L, LB, "pecnd"},
      {&out->omega_p, a.omega_p, E, L, LB, "omega_p"},
      {&out->phi, a.phi, E, L, LB, "phi"},
  };
  for (const Spec& sp : specs)
    if (encode_tma_map(sp.m, sp.base, sp.slices, sp.rows, sp.box, sp.name, err, errlen)) return 1;
  return 0;
}

bool fused_supports(int nlev) { return instance_for(nlev) > 0; }

int fused_instance_levels(int nlev) { return instance_for(nlev); }
int fused_instance_cluster(int nlev) { return instance_for(nlev) ? cluster_for(instance_for(nlev)) : 0; }

cudaError_t launch_fused(const KernelArgs& a0, cudaStream_t s) {
  KernelArgs a = a0;
  // distance: nlev=72 (CTA triples) -> 74 elements (16: 0.921, 32: 0.937, 74: 0.946, 148: 0.944 of the measured peak);
  // nlev=128 (CTA pairs) -> 32 (flat optimum 4...48, 0.74 at 148). Sweeps: profiles/README.md.
  // A caller's pf_dist < 0 turns the prefetch off (the zero-copy host path).
  a.pf_dist = a0.pf_dist < 0 ? 0 : (a.nlev == 72 ? sm_count() / 2 : 32);  // 74 on a 148-SM B200
  switch (instance_for(a.nlev)) {
    case 72: return launch_nlev<72>(a, s);
    case 128: return launch_nlev<128>(a, s);
    case 0: return cudaErrorInvalidValue;
  }
  return launch_fused_more(a, s);
}

}  // namespace caar
