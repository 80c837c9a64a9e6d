// Slab-partitioned MatMult_Elliptic (elliptic.C:297-339) over 2/4/8 GPUs: the grid is cut along its
// outermost axis, one process per GPU.  Derivatives along the local axes never leave the GPU.  The
// axis-0 chain  D_0 (eta D_0 w + eta' w g0)  runs on "pencils" (all P planes of 1/G of the lines):
// a stage kernel (elliptic_persist.cu) pads the local input and pushes each plane's lines into the
// owning rank's pencil with contiguous stores over NVLink (the forward all-to-all); the persistent chain
// kernel, launched behind it, runs the local-axis items while those arrive, then the pencil items out of
// local memory, whose epilogue stores the result rows straight into the plane owners' partial field (the
// backward all-to-all), then the last-axis items, which read part[0] after DONE.  Ranks order themselves
// with two epoch flags in peer memory (READY: my planes are in your pencil; DONE: all my results are in
// your partial field), never through the host.
#include "../../include/spectral_b200.h"
#include "common.cuh"
#include "deriv.h"
#include "elliptic.h"
#include "persist.h"

namespace sb200 {

namespace {

struct PeerPtrs {
  const double* x[SB200_MAX_RANKS];
};

__global__ void slab_to_pencil_kernel(PeerPtrs pp, double* __restrict__ xp, int P, int nloc, long long R0, long long Rp,
                                      int rank) {
  const long long total = (long long)P * Rp, stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int m = (int)(i / Rp);
    const long long nl = i - (long long)m * Rp;
    const int q = m / nloc;
    xp[i] = __ldcg(pp.x[q] + (long long)(m - q * nloc) * R0 + (long long)rank * Rp + nl);
  }
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// One descriptor per rank: its part[0] field as a 2-D fp64 tensor [nloc planes][R0 lines], box = 8 lines x nloc planes (the rows
// of one pencil item that land on that rank).  Returns false when the driver offers no TMA descriptor API (the kernel then keeps
// its per-thread stores).
bool encode_part0_maps(double* const* part0peer, int G, long long R0, int nloc, SlabMaps* out) {
  static EncodeTiledFn encode = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qr) == cudaSuccess && qr == cudaDriverEntryPointSuccess)
      encode = (EncodeTiledFn)fn;
    else
      cudaGetLastError();
  }
  if (!encode || nloc > 256) return false;
  for (int q = 0; q < G; q++) {
    const cuuint64_t gdim[2] = {(cuuint64_t)R0, (cuuint64_t)nloc};
    const cuuint64_t gstr[1] = {(cuuint64_t)R0 * sizeof(double)};
    const cuuint32_t box[2] = {8u, (cuuint32_t)nloc};
    const cuuint32_t es[2] = {1u, 1u};
    if (encode(&out->m[q], CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, (void*)part0peer[q], gdim, gstr, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return false;
  }
  return true;
}

int ilog2(int v) {
  int l = 0;
  while ((1 << l) < v) l++;
  return l;
}

}  // namespace

int slab_to_pencil(const SymmArena& a, const double* x_slab, double* x_pencil, int P, long long R0, cudaStream_t s) {
  PeerPtrs pp;
  for (int q = 0; q < SB200_MAX_RANKS; q++) pp.x[q] = q < a.nranks ? a.on(q, x_slab) : nullptr;
  const long long Rp = R0 / a.nranks, total = (long long)P * Rp;
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  slab_to_pencil_kernel<<<(unsigned)blocks, 256, 0, s>>>(pp, x_pencil, P, P / a.nranks, R0, Rp, a.rank);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return 0;
}

int EllipticCtx::refresh_pencils(cudaStream_t s) {
  // collective: every rank reaches this at the same point (first MatMult after a FormFunction)
  SB_TRY(arena.barrier(s));
  const int P = gdim[0];
  SB_TRY(slab_to_pencil(arena, eta, eta_p, P, gd.stride[0], s));
  SB_TRY(slab_to_pencil(arena, deta, deta_p, P, gd.stride[0], s));
  SB_TRY(slab_to_pencil(arena, gradu[0], g0_p, P, gd.stride[0], s));
  pencil_valid = true;
  return 0;
}

void free_slab_maps(SlabMaps* m) { delete m; }

bool elliptic_slab_fused_supported(const EllipticCtx& e) {
  const int d = e.gd.d, G = e.arena.nranks;
  if (G < 2 || d < 2) return false;
  const int P = e.gdim[0];
  for (int j = 1; j < d; j++)
    if (e.gdim[j] != P) return false;
  if (!(P == 32 || P == 64 || P == 128)) return false;
  if ((G & (G - 1)) != 0 || P % G != 0) return false;
  const long long R0 = e.gd.stride[0];
  if (R0 % G != 0 || (R0 / G) % 16 != 0) return false;
  return (e.gd.m / P) % 16 == 0;
}

int elliptic_matmult_slab_fused(EllipticCtx& e, const double* U, double* V, cudaStream_t s) {
  SB_CHECK(e.arena.attached(), SB200_ERR_USER, "slab partition: peers are not attached (exchange the IPC handles first)");
  const int P = e.gdim[0], d = e.gd.d, G = e.arena.nranks;
  if (!e.sync) {
    SB_CUDA(cudaMalloc((void**)&e.sync, 512));
    SB_CUDA(cudaMemsetAsync(e.sync, 0, 512, s));
  }
  if (!e.pencil_valid) SB_TRY(e.refresh_pencils(s));
  const unsigned long long epoch = ++e.mm_epoch;
  SymmFlags sf;
  for (int q = 0; q < SB200_MAX_RANKS; q++) sf.f[q] = q < G ? e.arena.flags(q) : nullptr;
  sf.rank = e.arena.rank;
  sf.nranks = G;
  PersistParams p = {};
  p.Ae = e.Dax[0]->d_Ae;
  p.Bo = e.Dax[0]->d_Bo;
  p.U = U;
  p.eta = e.eta;
  p.deta = e.deta;
  p.V = V;
  p.nlines = e.gd.m / P;
  p.d = d;
  for (int k = 0; k < d; k++) {
    p.g0[k] = e.gradu[k];
    p.part[k] = e.w[1 + k];
    p.R[k] = e.gd.stride[k];
  }
  p.sync = e.sync;
  p.sg.i0 = e.gd.i0;
  p.sg.n0g = e.gd.n0g;
  p.sg.goff = e.gd.goff;
  p.first_axis = 1;
  p.nranks = G;
  p.rank = e.arena.rank;
  const int nloc = P / G;
  p.lognloc = ilog2(nloc);
  for (int q = 0; q < G; q++) {
    p.part0peer[q] = e.arena.on(q, e.w[1]);
    p.wppeer[q] = e.arena.on(q, e.Wp);
  }
  p.Wp = e.Wp;
  p.eta_p = e.eta_p;
  p.deta_p = e.deta_p;
  p.g0_p = e.g0_p;
  p.R0 = e.gd.stride[0];
  p.Rp = p.R0 / G;
  p.sf = sf;
  p.epoch = epoch;
  // pencil results through TMA tensor stores (per-thread 16-byte peer stores when the descriptors cannot be encoded)
  if (!e.tmaps_tried) {
    e.tmaps_tried = true;
    e.tmaps = new SlabMaps();
    if (!encode_part0_maps(p.part0peer, G, p.R0, nloc, e.tmaps)) {
      delete e.tmaps;
      e.tmaps = nullptr;
    }
  }
  p.maps = e.tmaps;
  p.bulk = p.maps ? 1 : 0;
  p.trace = nullptr;
  return persist_run(P, p, s);
}

}  // namespace sb200
