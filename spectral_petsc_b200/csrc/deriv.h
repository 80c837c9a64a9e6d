// Internal interface of the generic per-axis derivative kernel (deriv_generic.cu).
#pragma once
#include <cuda_runtime.h>

namespace sb200 {

enum DerivMode { DERIV_STORE = 0, DERIV_SUB = 1, DERIV_ADD = 2 };

#define SB200_EO_MAX_JOBS 6
// The fused pad (loader gathers from the global vector) pays on launch-bound grids; beyond this many nodes the padded copy + 16-byte
// block loads are faster (measured at 128^3: 145 us fused against 26 + 100 us, profiles/r02_notes.md)
#define SB200_FUSE_PAD_MAX_NODES (1ll << 18)
// Likewise the fused crop-sum epilogue (its term loads are dependent L2 round trips of the finishing job's warps): 180 us against
// 100 + 55 us at 128^3 for the Stokes viscous tail; small grids gain the launch
#define SB200_FUSE_CROP_MAX_NODES (1ll << 18)
#ifndef SB200_MAX_RANKS
#define SB200_MAX_RANKS 8
#endif

// Grid geometry behind the lines of a job of the even-odd kernel (only needed by its fused pad / crop modes).
struct EoLineMap {
  int d = 0, nc = 1, axis = 0;
  int dim[SB200_EO_MAX_JOBS] = {1, 1, 1, 1, 1, 1};
  long long istride[SB200_EO_MAX_JOBS] = {0, 0, 0, 0, 0, 0};  // strides of the interior (dim - 2) grid = the walk order of the global vector
};

struct DerivParams {
  const double* D;    // device, Pp x Pp row-major, zero padded
  const double* Ae = nullptr;  // even-odd halves of D zero padded to HP x HP (DiffMatrix::d_Aep / d_Bop, any P <= SB200_EO_MAX_P);
  const double* Bo = nullptr;  // with `sync` they enable the even-odd persistent kernel (deriv_eo.cu)
  int HP = 0;
  unsigned* sync = nullptr;    // 3 zero-initialised counters owned by the calling context (ticket, exited warps, finished items)
  int P, Pp;          // extent of the differentiated axis, padded extent (multiple of 32)
  const double* x;    // input field
  double* y;          // output field (must not alias x)
  const double* yin;  // accumulation input for SUB/ADD (may alias y, may be null = 0)
  long long O, R;     // array factored as (O, P, R), row-major
  int xs, xoff;       // element e of x lives at x[e*xs + xoff]  (AoS component access)
  int ys, yoff;       // same for y / yin
  int mode;           // DerivMode: y = acc | yin - acc | yin + acc
  int inplace_ok = 0; // internal callers of the even-odd kernel may pass y == x: an item reads its 8 lines completely before it writes them
  // Slab-partitioned axis (multi-GPU, O == 1): input row k is read from xpeer[k / nloc] at local row
  // k % nloc (peer memory over NVLink, the "all-gather" is the operand load itself); this rank computes
  // output rows [row0, row0 + nloc) and stores them at local rows 0..nloc-1.  npeer <= 1: off.
  int npeer = 0, nloc = 0, row0 = 0;
  const double* xpeer[8] = {};

  // ---- fused scatters (even-odd kernel only, single GPU) -------------------------------------------------------------------
  // The job's lines are the lines along `lm.axis` of a (lm.d-dimensional grid) x (lm.nc trailing components) array, in row-major
  // order with the component fastest - the (O, P, R) factorisation above with R = stride[axis] * nc.
  EoLineMap lm = {};
  // Fused pad (the VecScatter global -> local of stokes.C:635-637 / elliptic.C:305-308 with zero Dirichlet rows): when gsrc is
  // set, x is ignored and element (node, comp) is gsrc[gid(node) * gs_stride + gs_off + comp] at interior nodes, 0 on the boundary.
  const double* gsrc = nullptr;
  int gs_stride = 0, gs_off = 0;
  // Fused crop (the VecScatter local -> global of stokes.C:592,617,673 together with the VecAXPY chain that precedes it): when
  // gdst is set, y / yin / mode are ignored and interior elements go to gdst[gid * gd_stride + gd_off + comp]:
  //   fin == EO_FIN_SUM : ((0 + sign*T_0) + sign*T_1 ...) + sign*(D x), T_t = term[t] (fields of the layout y would have, written
  //                       by EARLIER jobs of the same launch: the kernel orders them), nterms < SB200_EO_MAX_JOBS; then, if
  //                       (sub), v = v + (-1) * sub[same index]                               (crop_sum_kernel / crop_kernel)
  //   fin == EO_FIN_RAW : v = D x; if (add) v = gdst + v; if (sub) v = v + (-1) * sub[same index]           (crop_nodes_kernel)
  double* gdst = nullptr;
  int gd_stride = 0, gd_off = 0, fin = 0, nterms = 0, add = 0;
  int self_pos = -1;  // EO_FIN_SUM: the job's own value enters the chain after self_pos terms (-1 = last, i.e. after all of them), so any
                      // axis can be the one that finishes the sum while the chain keeps the reference's axis order
  const double* term[SB200_EO_MAX_JOBS - 1] = {};
  const double* sub = nullptr;
  double sign = 1.0;
  // Backward all-to-all of the slab partition folded into the epilogue of the PENCIL derivative (O == 1, R = Rp columns, unit strides,
  // DERIV_STORE or "0 - D x"): row m of the result belongs to rank m / peer_nloc and is stored straight into that rank's field,
  // ypeer[q][(m - q*peer_nloc) * peer_R + peer_col0 + column]  (16-byte stores over NVLink), so no push kernel re-reads a pencil buffer.
  double* ypeer[SB200_MAX_RANKS] = {};
  int peer_on = 0, peer_nloc = 0, peer_negate = 0;
  long long peer_R = 0, peer_col0 = 0;
};
enum { EO_FIN_NONE = 0, EO_FIN_SUM = 1, EO_FIN_RAW = 2 };

int deriv_apply(const DerivParams& p, cudaStream_t stream);
bool deriv_eo_supported(const DerivParams& p);
int deriv_eo_apply(const DerivParams& p, unsigned* sync, cudaStream_t stream);
// Up to SB200_EO_MAX_JOBS derivatives sharing the matrix (same extent) in ONE launch; outputs must be distinct.
int deriv_eo_batch(const DerivParams* jobs, int n, unsigned* sync, cudaStream_t stream);
// The same for jobs that may differ in extent: one launch when they all share the matrix, else one launch per job in order
// (a job's terms then come from earlier launches).
int deriv_eo_jobs(const DerivParams* jobs, int n, unsigned* sync, cudaStream_t stream);

void count_launch(int n = 1);

struct SymmArena;
// Transpose-based derivative along the partitioned axis of a slab-distributed field (slab_deriv.cu).
bool slab_deriv0_pencil_supported(const SymmArena& a, const DerivParams& p);
int slab_deriv0_pencil(SymmArena& a, const DerivParams& p, int nloc, int i0, double* Xp, double* Yp, cudaStream_t s);

}  // namespace sb200
