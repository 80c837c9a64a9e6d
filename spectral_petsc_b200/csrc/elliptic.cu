// Elliptic operator shells: MatMult_Elliptic (elliptic.C:297-339) and FormFunction
// (elliptic.C:481-533) on device-resident fp64 vectors, arbitrary dimension.
//
// Generic path (any rank / extents): structured pad (scatterGL + scatterDL as index arithmetic,
// no index arrays), one DMMA derivative launch per axis, one pointwise flux kernel, one
// derivative launch per axis with the "-=" accumulation fused in its epilogue, structured crop.
// The 3-D fused plane kernels (elliptic_fused.cu) replace the middle of this when enabled.
#include "elliptic.h"

#include <algorithm>
#include <cmath>
#include <vector>

#include "../../include/spectral_b200.h"
#include "cheb_matrix.h"
#include "common.cuh"
#include "deriv.h"

namespace sb200 {

namespace {

// Line-based pad / crop: one (ty) thread row per grid line of the LAST axis, so the d-1 leading
// indices are decoded once per line and the walk along the line is contiguous in both vectors.
struct LineInfo {
  bool interior;   // all leading indices interior
  long long gid0;  // global id of the line's first interior node (k = 1)
  long long did0;  // dirichlet id of the line's first node (k = 0)
};

__device__ __forceinline__ LineInfo decode_line(const GridDesc& gd, long long line) {
  // Same walk-order semantics as SetupBC (elliptic.C:386-415), specialised to whole last-axis lines.
  // Slab view: axis-0 indices are offset by gd.i0 inside a global extent gd.n0g and the ordinals are
  // relative to the first locally stored interior / boundary node.
  const int d = gd.d, PL = gd.dim[d - 1];
  long long rem = line, cnt = -gd.goff;
  bool prefix_int = true;
  for (int j = 0; j < d - 1; j++) {
    const long long s = gd.stride[j] / PL;
    const int il = (int)(rem / s);
    rem -= (long long)il * s;
    const int i = gd.gidx(j, il), ext = gd.gext(j);
    const bool b = (i == 0) || (i == ext - 1);
    if (prefix_int) {
      int c = i - 1;
      c = c < 0 ? 0 : (c > ext - 2 ? ext - 2 : c);
      cnt += (long long)c * gd.istride[j];
      if (b) prefix_int = false;
    }
  }
  LineInfo li;
  li.interior = prefix_int;
  li.gid0 = cnt;                 // interior nodes before this line
  li.did0 = line * PL - cnt;     // boundary nodes before this line
  return li;
}

__global__ void pad_kernel(GridDesc gd, long long nlines, const double* __restrict__ U,
                           const double* __restrict__ dir, double* __restrict__ w0) {
  // one thread row (threadIdx.y) per line; the line decode is done once per row by lane 0
  const long long line = (long long)blockIdx.x * blockDim.y + threadIdx.y;
  const bool live = line < nlines;
  const int PL = gd.dim[gd.d - 1];
  __shared__ LineInfo sli[32];
  if (threadIdx.x == 0 && live) sli[threadIdx.y] = decode_line(gd, line);
  __syncthreads();
  if (!live) return;
  const LineInfo li = sli[threadIdx.y];
  double* wl = w0 + line * PL;
  for (int k = threadIdx.x; k < PL; k += blockDim.x) {
    double v;
    if (li.interior && k > 0 && k < PL - 1) v = U[li.gid0 + k - 1];
    else if (!dir) v = 0.0;
    else if (!li.interior) v = dir[li.did0 + k];
    else v = dir[li.did0 + (k == 0 ? 0 : 1)];
    wl[k] = v;
  }
}

__global__ void crop_kernel(GridDesc gd, long long nlines, const double* __restrict__ w0,
                            const double* __restrict__ b, double* __restrict__ V) {
  const long long line = (long long)blockIdx.x * blockDim.y + threadIdx.y;
  if (line >= nlines) return;
  const int PL = gd.dim[gd.d - 1];
  const LineInfo li = decode_line(gd, line);
  if (!li.interior) return;
  const double* wl = w0 + line * PL;
  for (int k = 1 + threadIdx.x; k < PL - 1; k += blockDim.x) {
    double v = wl[k];
    const long long gid = li.gid0 + k - 1;
    if (b) v = v + (-1.0) * b[gid];  // VecAXPY(rhs, -1.0, ac->b) elliptic.C:530
    V[gid] = v;
  }
}

struct FluxPtrs {
  double* w[SB200_MAX_DIM];
  const double* g0[SB200_MAX_DIM];
};

// elliptic.C:319-323: w[d] = eta*w[d] + deta*u*gradu[d]
__global__ void flux_kernel(long long m, int d, const double* __restrict__ u, const double* __restrict__ eta,
                            const double* __restrict__ deta, FluxPtrs fp) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += stride) {
    const double e = eta[i], de = deta[i], ui = u[i];
    for (int k = 0; k < d; k++) {
      fp.w[k][i] = __dadd_rn(__dmul_rn(e, fp.w[k][i]), __dmul_rn(__dmul_rn(de, ui), fp.g0[k][i]));
    }
  }
}

// The same with u taken from the GLOBAL vector (zero on the boundary): the fused generic path never materialises the padded field.
__global__ void flux_global_kernel(GridDesc gd, int d, const double* __restrict__ U, const double* __restrict__ eta,
                                   const double* __restrict__ deta, FluxPtrs fp) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  const int PL = gd.dim[d - 1];
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < gd.m; i += stride) {
    const long long line = i / PL;
    const int k = (int)(i - line * PL);
    const LineInfo li = decode_line(gd, line);
    const double ui = (li.interior && k > 0 && k < PL - 1) ? U[li.gid0 + k - 1] : 0.0;
    const double e = eta[i], de = deta[i];
    for (int q = 0; q < d; q++) {
      fp.w[q][i] = __dadd_rn(__dmul_rn(e, fp.w[q][i]), __dmul_rn(__dmul_rn(de, ui), fp.g0[q][i]));
    }
  }
}

// elliptic.C:507-513: eta = 1 + gamma*pow(u,p); deta = p*gamma*pow(u,p-1); w[d] = eta*gradu[d]
__global__ void coef_flux_kernel(long long m, int d, double gamma, double expo, const double* __restrict__ u,
                                 double* __restrict__ eta, double* __restrict__ deta, FluxPtrs fp) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += stride) {
    const double ui = u[i];
    const double e = __dadd_rn(1.0, __dmul_rn(gamma, pow(ui, expo)));
    const double de = __dmul_rn(__dmul_rn(expo, gamma), pow(ui, expo - 1.0));
    eta[i] = e;
    deta[i] = de;
    for (int k = 0; k < d; k++) fp.w[k][i] = __dmul_rn(e, fp.g0[k][i]);
  }
}

int grid_for(long long n) {
  long long b = (n + 255) / 256;
  return (int)std::min<long long>(b, 148 * 16);
}

}  // namespace

// ---- derivative-matrix cache -------------------------------------------------------------
int DiffMatrix::create(int P, DiffMatrix* out) {
  out->P = P;
  out->Pp = (P + 31) / 32 * 32;
  std::vector<double> D = cgl_diff_matrix(P);
  std::vector<double> Dp((size_t)out->Pp * out->Pp, 0.0);
  for (int i = 0; i < P; i++)
    for (int j = 0; j < P; j++) Dp[(size_t)i * out->Pp + j] = D[(size_t)i * P + j];
  SB_CUDA(cudaMalloc((void**)&out->d_D, Dp.size() * sizeof(double)));
  SB_CUDA(cudaMemcpy(out->d_D, Dp.data(), Dp.size() * sizeof(double), cudaMemcpyHostToDevice));
  if (P % 2 == 0) {
    std::vector<double> Ae, Bo;
    cgl_even_odd(P, Ae, Bo);
    SB_CUDA(cudaMalloc((void**)&out->d_Ae, Ae.size() * sizeof(double)));
    SB_CUDA(cudaMalloc((void**)&out->d_Bo, Bo.size() * sizeof(double)));
    SB_CUDA(cudaMemcpy(out->d_Ae, Ae.data(), Ae.size() * sizeof(double), cudaMemcpyHostToDevice));
    SB_CUDA(cudaMemcpy(out->d_Bo, Bo.data(), Bo.size() * sizeof(double), cudaMemcpyHostToDevice));
  }
  if (P <= SB200_EO_MAX_P) {
    out->HP = ((P + 1) / 2 + 7) / 8 * 8;
    std::vector<double> Ae, Bo;
    cgl_even_odd_padded(P, out->HP, Ae, Bo);
    SB_CUDA(cudaMalloc((void**)&out->d_Aep, Ae.size() * sizeof(double)));
    SB_CUDA(cudaMalloc((void**)&out->d_Bop, Bo.size() * sizeof(double)));
    SB_CUDA(cudaMemcpy(out->d_Aep, Ae.data(), Ae.size() * sizeof(double), cudaMemcpyHostToDevice));
    SB_CUDA(cudaMemcpy(out->d_Bop, Bo.data(), Bo.size() * sizeof(double), cudaMemcpyHostToDevice));
  }
  return 0;
}

void DiffMatrix::destroy() {
  if (d_D) cudaFree(d_D);
  if (d_Ae) cudaFree(d_Ae);
  if (d_Bo) cudaFree(d_Bo);
  if (d_Aep) cudaFree(d_Aep);
  if (d_Bop) cudaFree(d_Bop);
  d_D = d_Ae = d_Bo = d_Aep = d_Bop = nullptr;
}

int GridDesc::init(int d_, const int* dim_) {
  SB_CHECK(d_ >= 1 && d_ <= SB200_MAX_DIM, SB200_ERR_USER, "dimension count must be in [1,10] (elliptic.C:138)");
  d = d_;
  m = 1;
  g = 1;
  for (int j = 0; j < d; j++) {
    SB_CHECK(dim_[j] >= 3, SB200_ERR_USER, "each extent must be >= 3 (needs an interior node)");
    dim[j] = dim_[j];
  }
  for (int j = d - 1; j >= 0; j--) {
    stride[j] = m;
    istride[j] = g;
    m *= dim[j];
    g *= dim[j] - 2;
  }
  i0 = 0;
  n0g = dim[0];
  goff = 0;
  return 0;
}

int GridDesc::init_slab(int d_, const int* dim_global, int rank, int nranks) {
  SB_TRY(init(d_, dim_global));
  if (nranks == 1) return 0;
  SB_CHECK(d >= 2, SB200_ERR_USER, "slab partition needs at least two axes");
  SB_CHECK(dim[0] % nranks == 0, SB200_ERR_USER, "slab partition: the outermost extent must be divisible by the number of ranks");
  const int nloc = dim[0] / nranks;
  n0g = dim[0];
  i0 = rank * nloc;
  dim[0] = nloc;
  m = (long long)nloc * stride[0];
  // interior planes among [i0, i0 + nloc)
  const int lo = i0 < 1 ? 1 : i0, hi = (i0 + nloc > n0g - 1) ? n0g - 1 : i0 + nloc;  // [lo, hi)
  g = (long long)(hi > lo ? hi - lo : 0) * istride[0];
  goff = (long long)(lo - 1) * istride[0];
  return 0;
}

// ---- EllipticCtx ---------------------------------------------------------------------------
int EllipticCtx::create(int d, const int* dim, int rank, int nranks, EllipticCtx** out) {
  EllipticCtx* e = new EllipticCtx();
  int rc = e->init(d, dim, rank, nranks);
  if (rc) {
    delete e;
    return rc;
  }
  *out = e;
  return 0;
}

int EllipticCtx::init(int d, const int* dim, int rank, int nranks) {
  SB_TRY(gd.init_slab(d, dim, rank, nranks));
  gtot = 1;
  for (int k = 0; k < d; k++) {
    gdim[k] = dim[k];
    gtot *= dim[k] - 2;
  }
  nw = 2 + d;  // elliptic.C:259
  const size_t mb = (size_t)gd.m * sizeof(double);
  // every exchangeable array comes from one peer-mapped arena, in the same order on every rank
  const int narr = nw + d + 2 + (nranks > 1 ? 6 : 0);
  SB_TRY(arena.init((size_t)narr * (mb + 256), rank, nranks));
  for (int k = 0; k < nw; k++) SB_CHECK((w[k] = arena.alloc_doubles(gd.m)), SB200_ERR_CUDA, "arena exhausted");
  for (int k = 0; k < d; k++) {
    SB_CHECK((gradu[k] = arena.alloc_doubles(gd.m)), SB200_ERR_CUDA, "arena exhausted");
    SB_CUDA(cudaMemset(gradu[k], 0, mb));
  }
  SB_CHECK((eta = arena.alloc_doubles(gd.m)), SB200_ERR_CUDA, "arena exhausted");
  SB_CHECK((deta = arena.alloc_doubles(gd.m)), SB200_ERR_CUDA, "arena exhausted");
  if (nranks > 1) {
    SB_CHECK((eta_p = arena.alloc_doubles(gd.m)), SB200_ERR_CUDA, "arena exhausted");
    SB_CHECK((deta_p = arena.alloc_doubles(gd.m)), SB200_ERR_CUDA, "arena exhausted");
    SB_CHECK((g0_p = arena.alloc_doubles(gd.m)), SB200_ERR_CUDA, "arena exhausted");
    SB_CHECK((Wp = arena.alloc_doubles(gd.m)), SB200_ERR_CUDA, "arena exhausted");
    SB_CHECK((Xp = arena.alloc_doubles(gd.m)), SB200_ERR_CUDA, "arena exhausted");
    SB_CHECK((Yp = arena.alloc_doubles(gd.m)), SB200_ERR_CUDA, "arena exhausted");
  }
  SB_CUDA(cudaMalloc((void**)&sync, 512));
  SB_CUDA(cudaMemset(sync, 0, 512));
  SB_CUDA(cudaMalloc((void**)&dirichlet, std::max<size_t>(8, (size_t)(gd.m - gd.g) * sizeof(double))));
  SB_CUDA(cudaMemset(dirichlet, 0, std::max<size_t>(8, (size_t)(gd.m - gd.g) * sizeof(double))));
  SB_CUDA(cudaMalloc((void**)&b, std::max<size_t>(8, (size_t)gd.g * sizeof(double))));
  SB_CUDA(cudaMemset(b, 0, std::max<size_t>(8, (size_t)gd.g * sizeof(double))));
  {  // VecSet(eta, 1.0); VecSet(deta, 0.0) elliptic.C:266-267
    std::vector<double> ones((size_t)gd.m, 1.0);
    SB_CUDA(cudaMemcpy(eta, ones.data(), mb, cudaMemcpyHostToDevice));
    SB_CUDA(cudaMemset(deta, 0, mb));
  }
  for (int k = 0; k < d; k++) {
    Dax[k] = nullptr;
    for (int q = 0; q < k; q++)
      if (gdim[q] == gdim[k]) Dax[k] = Dax[q];
    if (!Dax[k]) {
      DiffMatrix* dm = new DiffMatrix();
      SB_TRY(DiffMatrix::create(gdim[k], dm));
      owned.push_back(dm);
      Dax[k] = dm;
    }
  }
  return 0;
}

EllipticCtx::~EllipticCtx() {
  free_slab_maps(tmaps);
  arena.destroy();
  if (dirichlet) cudaFree(dirichlet);
  if (b) cudaFree(b);
  if (sync) cudaFree(sync);
  if (gexec) {
    cudaDeviceSynchronize();  // a replay may still be in flight
    cudaGraphExecDestroy(gexec);
  }
  if (gstream) cudaStreamDestroy(gstream);
  if (gU) cudaFree(gU);
  if (gV) cudaFree(gV);
  for (DiffMatrix* dm : owned) {
    dm->destroy();
    delete dm;
  }
}

// Single GPU, rank <= SB200_EO_MAX_JOBS, every extent within the even-odd kernel's reach: the generic path runs as
// [gradient batch with the pad in its loader] -> flux -> [divergence batch with the "-=" chain and the crop in its epilogue].
bool EllipticCtx::fusable() const {
  if (arena.nranks > 1 || gd.d > SB200_EO_MAX_JOBS) return false;
  for (int k = 0; k < gd.d; k++)
    if (!deriv_eo_supported(job(k, w[0], w[1], nullptr, DERIV_STORE))) return false;
  return true;
}

EoLineMap EllipticCtx::line_map(int axis) const {
  EoLineMap lm;
  lm.d = gd.d;
  lm.nc = 1;
  lm.axis = axis;
  for (int j = 0; j < gd.d; j++) {
    lm.dim[j] = gd.dim[j];
    lm.istride[j] = gd.istride[j];
  }
  return lm;
}

DerivParams EllipticCtx::job(int axis, const double* x, double* y, const double* yin, int mode) const {
  DerivParams p;
  p.D = Dax[axis]->d_D;
  p.Ae = Dax[axis]->d_Aep;
  p.Bo = Dax[axis]->d_Bop;
  p.HP = Dax[axis]->HP;
  p.sync = sync + 10;  // counters of the even-odd derivative kernel ([0..5]: persistent chain phases, [8]: stage)
  p.P = Dax[axis]->P;
  p.Pp = Dax[axis]->Pp;
  p.x = x;
  p.y = y;
  p.yin = yin;
  p.O = gd.m / (gd.stride[axis] * gd.dim[axis]);
  p.R = gd.stride[axis];
  p.xs = p.ys = 1;
  p.xoff = p.yoff = 0;
  p.mode = mode;
  return p;
}

// The divergence half of both shells on the fused path: T_k = D_k w[1+k] in place for k < d-1, the last axis' epilogue forms
// ((0 - T_0) - T_1 ...) - D_{d-1} w[d] (elliptic.C:329-334 / 520-524), subtracts rhs when given (:530) and scatters (:336-337).
int EllipticCtx::fused_tail(const double* rhs, double* V, cudaStream_t s) {
  const int d = gd.d;
  DerivParams jobs[SB200_EO_MAX_JOBS];
  for (int k = 0; k < d - 1; k++) {
    jobs[k] = job(k, w[1 + k], w[1 + k], nullptr, DERIV_STORE);
    jobs[k].inplace_ok = 1;
  }
  DerivParams& f = jobs[d - 1] = job(d - 1, w[d], nullptr, nullptr, DERIV_STORE);
  f.lm = line_map(d - 1);
  f.gdst = V;
  f.gd_stride = 1;
  f.gd_off = 0;
  f.fin = EO_FIN_SUM;
  f.nterms = d - 1;
  for (int k = 0; k < d - 1; k++) f.term[k] = w[1 + k];
  f.sign = -1.0;
  f.sub = rhs;
  return deriv_eo_jobs(jobs, d, sync + 10, s);
}

int EllipticCtx::deriv(int axis, const double* x, double* y, const double* yin, int mode, cudaStream_t s) {
  DerivParams p;
  p.D = Dax[axis]->d_D;
  p.Ae = Dax[axis]->d_Aep;
  p.Bo = Dax[axis]->d_Bop;
  p.HP = Dax[axis]->HP;
  p.sync = sync + 10;  // counters of the even-odd derivative kernel ([0..5]: persistent chain phases, [8]: stage)
  p.P = Dax[axis]->P;
  p.Pp = Dax[axis]->Pp;
  p.x = x;
  p.y = y;
  p.yin = yin;
  p.O = gd.m / (gd.stride[axis] * gd.dim[axis]);
  p.R = gd.stride[axis];
  p.xs = p.ys = 1;
  p.xoff = p.yoff = 0;
  p.mode = mode;
  if (axis == 0 && arena.nranks > 1) {
    // the partitioned axis: through the column pencils (two pushes over NVLink) when the columns divide by the
    // number of ranks; otherwise operand rows are pulled from the planes' owners (x must be an arena array) and the
    // barriers order the peers' writes of x before our reads and our reads before their next writes
    SB_CHECK(arena.attached(), SB200_ERR_USER, "slab partition: peers are not attached (exchange the IPC handles first)");
    if (slab_deriv0_pencil_supported(arena, p)) return slab_deriv0_pencil(arena, p, gd.dim[0], gd.i0, Xp, Yp, s);
    p.npeer = arena.nranks;
    p.nloc = gd.dim[0];
    p.row0 = gd.i0;
    for (int q = 0; q < arena.nranks; q++) p.xpeer[q] = arena.on(q, x);
    SB_TRY(arena.barrier(s));
    SB_TRY(deriv_apply(p, s));
    return arena.barrier(s);
  }
  return deriv_apply(p, s);
}

int EllipticCtx::pad(const double* U, bool with_dirichlet, double* local, cudaStream_t s) {
  const int PL = gd.dim[gd.d - 1];
  const long long nlines = gd.m / PL;
  const int tx = 32;
  dim3 blk(tx, 256 / tx);
  pad_kernel<<<(unsigned)((nlines + blk.y - 1) / blk.y), blk, 0, s>>>(gd, nlines, U, with_dirichlet ? dirichlet : nullptr, local);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return 0;
}

int EllipticCtx::crop(const double* local, const double* rhs, double* V, cudaStream_t s) {
  const int PL = gd.dim[gd.d - 1];
  const long long nlines = gd.m / PL;
  const int tx = PL >= 128 ? 128 : (PL > 32 ? 64 : 32);
  dim3 blk(tx, 256 / tx);
  crop_kernel<<<(unsigned)((nlines + blk.y - 1) / blk.y), blk, 0, s>>>(gd, nlines, local, rhs, V);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return 0;
}

int EllipticCtx::matmult(const double* U, double* V, cudaStream_t s) {
  SB_CHECK(U && V && U != V, SB200_ERR_ARG, "MatMult_Elliptic: U and V must be distinct non-null vectors");
  if (arena.nranks > 1) {
    SB_CHECK(arena.attached(), SB200_ERR_USER, "slab partition: peers are not attached (exchange the IPC handles first)");
    SB_CHECK(!arena.failed(), SB200_ERR_CUDA, "slab partition: a device-side flag wait timed out earlier (a peer never arrived or the ranks' calls went out of step); results are undefined, the context refuses further work");
    if ((path == 0 || path == 3) && elliptic_slab_fused_supported(*this)) {
      last_kernel = "slab step: stage_kernel + persist_kernel<P,8,1,SLAB> per rank (axis-0 chain on pencils exchanged through NVLink peer memory)";
      return elliptic_matmult_slab_fused(*this, U, V, s);
    }
    SB_CHECK(path <= 1, SB200_ERR_SUP, "slab partition: the fused path needs equal extents P in {32,64,128}");
  } else if (path == 3 || (path == 0 && elliptic_persist_supported(*this))) {
    SB_CHECK(elliptic_persist_supported(*this), SB200_ERR_SUP, "persistent path needs equal extents P % 16 == 0 between 32 and 160");
    last_kernel = "persist_kernel<P,NWARPS,1,MW> phases A+B (the whole MatMult step: 2 PDL-linked launches; MW = 2 warps per item at P = 128)";
    return elliptic_matmult_persist(*this, U, V, s);
  }
  if (path == 2 && arena.nranks == 1) {
    SB_CHECK(elliptic_fused_supported(*this), SB200_ERR_SUP, "fused path needs equal extents P in {32,64,128}");
    last_kernel = "chain_kernel per axis";
    return elliptic_matmult_fused(*this, U, V, s);
  }
  if (path == 4 && arena.nranks == 1) {
    last_kernel = "generic path replayed from a CUDA graph";
    return matmult_graph(U, V, s);
  }
  last_kernel = "generic path: pad + per-axis deriv_kernel / eo_deriv_kernel + pointwise kernels";
  return matmult_generic(U, V, s);
}

int EllipticCtx::matmult_graph(const double* U, double* V, cudaStream_t s) {
  const size_t bytes = (size_t)gd.g * sizeof(double);
  if (!gexec) {
    if (!gU) SB_CUDA(cudaMalloc((void**)&gU, bytes));
    if (!gV) SB_CUDA(cudaMalloc((void**)&gV, bytes));
    if (!gstream) SB_CUDA(cudaStreamCreateWithFlags(&gstream, cudaStreamNonBlocking));
    SB_CUDA(cudaStreamSynchronize(s));  // the warm-up below uses the context's scratch fields on another stream
    SB_CUDA(cudaMemsetAsync(gU, 0, bytes, gstream));
    SB_TRY(matmult_generic(gU, gV, gstream));  // once outside the capture: function attributes, lazy module loading
    SB_CUDA(cudaStreamSynchronize(gstream));
    SB_CUDA(cudaStreamBeginCapture(gstream, cudaStreamCaptureModeThreadLocal));
    const int rc = matmult_generic(gU, gV, gstream);
    cudaGraph_t graph = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(gstream, &graph);
    if (rc || ce != cudaSuccess || !graph) {
      if (graph) cudaGraphDestroy(graph);
      cudaGetLastError();
      SB_CHECK(rc == 0, rc, "MatMult_Elliptic: the generic path failed while being captured");
      set_last_error(std::string("cudaStreamEndCapture: ") + cudaGetErrorString(ce));
      return SB200_ERR_CUDA;
    }
    size_t nn = 0;
    cudaGraphGetNodes(graph, nullptr, &nn);
    gnodes = (int)nn;
    const cudaError_t ie = cudaGraphInstantiate(&gexec, graph, 0);
    cudaGraphDestroy(graph);
    SB_CUDA(ie);
  }
  // the captured kernels read eta / deta / gradu through the context's own (fixed) arrays, so a new state needs no re-capture
  SB_CUDA(cudaMemcpyAsync(gU, U, bytes, cudaMemcpyDeviceToDevice, s));
  SB_CUDA(cudaGraphLaunch(gexec, s));
  SB_CUDA(cudaMemcpyAsync(V, gV, bytes, cudaMemcpyDeviceToDevice, s));
  count_launch(gnodes);
  return 0;
}

int EllipticCtx::matmult_generic(const double* U, double* V, cudaStream_t s) {
  const int d = gd.d;
  if (fusable()) {
    // 3 launches whatever the rank on small (launch-bound) grids: the gradient's loaders read U itself with the zero Dirichlet
    // rows filled in (:305-311); large grids keep the padded copy (4 launches)
    const bool fuse_pad = gd.m <= SB200_FUSE_PAD_MAX_NODES;
    if (!fuse_pad) SB_TRY(pad(U, false, w[0], s));
    DerivParams jobs[SB200_EO_MAX_JOBS];
    FluxPtrs fp;
    for (int k = 0; k < d; k++) {
      jobs[k] = job(k, fuse_pad ? nullptr : w[0], w[1 + k], nullptr, DERIV_STORE);
      if (fuse_pad) {
        jobs[k].lm = line_map(k);
        jobs[k].gsrc = U;
        jobs[k].gs_stride = 1;
        jobs[k].gs_off = 0;
      }
      fp.w[k] = w[1 + k];
      fp.g0[k] = gradu[k];
    }
    SB_TRY(deriv_eo_jobs(jobs, d, sync + 10, s));
    if (fuse_pad) flux_global_kernel<<<grid_for(gd.m), 256, 0, s>>>(gd, d, U, eta, deta, fp);  // :319-323
    else flux_kernel<<<grid_for(gd.m), 256, 0, s>>>(gd.m, d, w[0], eta, deta, fp);
    count_launch();
    SB_CUDA(cudaGetLastError());
    return fused_tail(nullptr, V, s);  // :329-337
  }
  SB_TRY(pad(U, false, w[0], s));                                              // :305-308
  for (int k = 0; k < d; k++) SB_TRY(deriv(k, w[0], w[1 + k], nullptr, DERIV_STORE, s));  // :309-311
  FluxPtrs fp;
  for (int k = 0; k < d; k++) {
    fp.w[k] = w[1 + k];
    fp.g0[k] = gradu[k];
  }
  flux_kernel<<<grid_for(gd.m), 256, 0, s>>>(gd.m, d, w[0], eta, deta, fp);  // :319-323
  count_launch();
  SB_CUDA(cudaGetLastError());
  // :329-334  w0 = 0; w0 -= D_k w[1+k] in axis order (the AXPY is the derivative's epilogue)
  for (int k = 0; k < d; k++) SB_TRY(deriv(k, w[1 + k], w[0], k == 0 ? nullptr : w[0], DERIV_SUB, s));
  SB_TRY(crop(w[0], nullptr, V, s));  // :336-337
  return 0;
}

int EllipticCtx::function(const double* U, double* F, cudaStream_t s) {
  SB_CHECK(U && F && U != F, SB200_ERR_ARG, "FormFunction: U and F must be distinct non-null vectors");
  const int d = gd.d;
  SB_TRY(pad(U, true, w[0], s));                                                   // :489-492
  const bool fused = fusable();
  if (fused) {
    DerivParams jobs[SB200_EO_MAX_JOBS];
    for (int k = 0; k < d; k++) jobs[k] = job(k, w[0], gradu[k], nullptr, DERIV_STORE);
    SB_TRY(deriv_eo_jobs(jobs, d, sync + 10, s));
  } else {
    for (int k = 0; k < d; k++) SB_TRY(deriv(k, w[0], gradu[k], nullptr, DERIV_STORE, s));  // :497-499
  }
  FluxPtrs fp;
  for (int k = 0; k < d; k++) {
    fp.w[k] = w[1 + k];
    fp.g0[k] = gradu[k];
  }
  coef_flux_kernel<<<grid_for(gd.m), 256, 0, s>>>(gd.m, d, gamma, exponent, w[0], eta, deta, fp);  // :506-513
  count_launch();
  SB_CUDA(cudaGetLastError());
  if (fused) {
    SB_TRY(fused_tail(b, F, s));  // :520-531
  } else {
    for (int k = 0; k < d; k++) SB_TRY(deriv(k, w[1 + k], w[0], k == 0 ? nullptr : w[0], DERIV_SUB, s));  // :520-524
    SB_TRY(crop(w[0], b, F, s));  // :528-531
  }
  pencil_valid = false;         // eta / deta / gradu[0] changed: the axis-0 pencil copies are stale
  return 0;
}

}  // namespace sb200
