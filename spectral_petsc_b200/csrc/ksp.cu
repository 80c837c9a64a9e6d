// Device-resident FGMRES(m) (ksp.h): every vector operation is a kernel on the caller's stream, the small
// Hessenberg / Givens work runs in one-thread kernels, and the host only reads one double per iteration (the
// recurrence residual norm, through mapped pinned memory) to take the convergence decision - the same
// decision point PETSc has.  Reductions are two-stage with a fixed summation order (deterministic), and on a
// slab partition the per-rank sums are combined through peer memory in rank order (identical on all ranks).
#include "ksp.h"

#include <cmath>
#include <cstring>

#include "../../include/spectral_b200.h"
#include "common.cuh"
#include "deriv.h"

namespace sb200 {

namespace {

constexpr int TPB = 256;

// The vector kernels of an Arnoldi step follow each other on one stream, each a few tens of microseconds long: launched as programmatic
// dependents, a kernel's blocks are set up while its predecessor drains and wait (griddepcontrol.wait) before their first global access.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_go() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = 0;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}
constexpr int SLOT = 64;     // doubles per all-reduce slot

__device__ __forceinline__ double block_sum(double v, double* sm) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) sm[warp] = v;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x == 0)
    for (int k = 0; k < TPB / 32; k++) t += sm[k];  // fixed order
  return t;  // valid on thread 0
}

// out[j] = sum_i x[i] * Y[j*ldy + i],  j in [0, nv).  grid = (nblocks, ceil(nv / CH)): x is read once per group of CH vectors.
template <int CH>
__global__ void __launch_bounds__(TPB) mdot_kernel(const double* __restrict__ x, const double* __restrict__ Y, long long ldy, int nv,
                                                   long long n, double* __restrict__ partial, unsigned* counters, double* __restrict__ out,
                                                   int vec2) {
  __shared__ double sm[TPB / 32];
  __shared__ bool last;
  pdl_go();
  pdl_wait();
  const int j0 = blockIdx.y * CH, cnt = min(CH, nv - j0);
  double acc[CH];
#pragma unroll
  for (int jj = 0; jj < CH; jj++) acc[jj] = 0.0;
  const long long stride = (long long)gridDim.x * TPB;
  if (vec2) {
    // 16-byte loads: every pointer is 16-byte aligned and ldy is even (checked on the host)
    const long long n2 = n >> 1;
    const double2* __restrict__ x2 = reinterpret_cast<const double2*>(x);
    for (long long i = (long long)blockIdx.x * TPB + threadIdx.x; i < n2; i += stride) {
      const double2 xi = x2[i];
#pragma unroll
      for (int jj = 0; jj < CH; jj++)
        if (jj < cnt) {
          const double2 yv = reinterpret_cast<const double2*>(Y + (long long)(j0 + jj) * ldy)[i];
          acc[jj] = fma(xi.x, yv.x, acc[jj]);
          acc[jj] = fma(xi.y, yv.y, acc[jj]);
        }
    }
    if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
      const double xi = x[n - 1];
#pragma unroll
      for (int jj = 0; jj < CH; jj++)
        if (jj < cnt) acc[jj] = fma(xi, Y[(long long)(j0 + jj) * ldy + n - 1], acc[jj]);
    }
  } else {
    for (long long i = (long long)blockIdx.x * TPB + threadIdx.x; i < n; i += stride) {
      const double xi = x[i];
#pragma unroll
      for (int jj = 0; jj < CH; jj++)
        if (jj < cnt) acc[jj] = fma(xi, Y[(long long)(j0 + jj) * ldy + i], acc[jj]);
    }
  }
#pragma unroll
  for (int jj = 0; jj < CH; jj++) {
    const double t = block_sum(acc[jj], sm);
    if (threadIdx.x == 0 && jj < cnt) partial[(long long)(j0 + jj) * gridDim.x + blockIdx.x] = t;
  }
  if (threadIdx.x == 0) {
    __threadfence();
    last = atomicAdd(counters + blockIdx.y, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (last) {
    // warp jj adds the per-block partials of vector j0+jj: lane-strided loads, then a shuffle tree (fixed order)
    __threadfence();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int jj = warp; jj < cnt; jj += TPB / 32) {
      double t = 0.0;
      for (unsigned b = lane; b < gridDim.x; b += 32) t += __ldcg(partial + (long long)(j0 + jj) * gridDim.x + b);
      for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
      if (lane == 0) out[j0 + jj] = t;
    }
    if (threadIdx.x == 0) counters[blockIdx.y] = 0;
  }
}

// Layout of the small-work array (doubles), m = restart:
//   H[(m+1)*m] | cs[m] | sn[m] | g[m+1] | y[m] | hcol[m+2] | scr[8]
struct SmallPtrs {
  double *H, *cs, *sn, *g, *y, *hcol, *scr;
  int m;
  __host__ __device__ static SmallPtrs make(double* base, int m) {
    SmallPtrs p;
    p.m = m;
    p.H = base;
    p.cs = p.H + (size_t)(m + 1) * m;
    p.sn = p.cs + m;
    p.g = p.sn + m;
    p.y = p.g + (m + 1);
    p.hcol = p.y + m;
    p.scr = p.hcol + (m + 2);
    return p;
  }
  static size_t count(int m) { return (size_t)(m + 1) * m + 2 * m + (m + 1) + m + (m + 2) + 8; }
};

struct HessArgs {  // on != 0: the block that finishes the norm also runs the Hessenberg / Givens update of column k
  SmallPtrs sp;
  int on, k;
  double* rnorm_dev;
  double* rnorm_host;
};
__device__ void hess_update(const SmallPtrs& p, int k, double* rnorm_dev, double* rnorm_host);

// y[i] += sign * sum_j c[j] * Y[j*ldy + i];  optionally out_nrm2 = sum_i y[i]^2 (of the updated y).
__global__ void __launch_bounds__(TPB) maxpy_kernel(double* __restrict__ y, const double* __restrict__ Y, long long ldy, int nv,
                                                    const double* __restrict__ c, double sign, long long n, double* __restrict__ partial,
                                                    unsigned* counter, double* __restrict__ out_nrm2, int vec2, HessArgs ha, int desc) {
  __shared__ double sm[TPB / 32];
  __shared__ double cs[64];
  __shared__ bool last;
  pdl_go();
  pdl_wait();
  if (threadIdx.x < nv) cs[threadIdx.x] = sign * c[threadIdx.x];
  __syncthreads();
  double acc = 0.0;
  const long long stride = (long long)gridDim.x * TPB;
  if (vec2) {
    // DESCENDING through the vectors: the multi-dot that ran just before walked them upwards, so the last ~100 MB it touched (the
    // high end of every vector) are still in the 126 MB L2 when this kernel starts there
    const long long n2 = n >> 1;
    double2* __restrict__ y2 = reinterpret_cast<double2*>(y);
    const long long first = (long long)blockIdx.x * TPB + threadIdx.x;
    const long long steps = first < n2 ? (n2 - 1 - first) / stride : -1;
    const long long istart = desc ? first + steps * stride : first, istep = desc ? -stride : stride;
    for (long long i = istart, c = 0; c <= steps; c++, i += istep) {
      double2 v = y2[i];
#pragma unroll 4
      for (int j = 0; j < nv; j++) {
        const double2 yv = reinterpret_cast<const double2*>(Y + (long long)j * ldy)[i];
        v.x = fma(cs[j], yv.x, v.x);
        v.y = fma(cs[j], yv.y, v.y);
      }
      y2[i] = v;
      acc = fma(v.x, v.x, acc);
      acc = fma(v.y, v.y, acc);
    }
    if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
      double v = y[n - 1];
      for (int j = 0; j < nv; j++) v = fma(cs[j], Y[(long long)j * ldy + n - 1], v);
      y[n - 1] = v;
      acc = fma(v, v, acc);
    }
  } else {
    for (long long i = (long long)blockIdx.x * TPB + threadIdx.x; i < n; i += stride) {
      double v = y[i];
      for (int j = 0; j < nv; j++) v = fma(cs[j], Y[(long long)j * ldy + i], v);
      y[i] = v;
      acc = fma(v, v, acc);
    }
  }
  if (!out_nrm2) return;
  const double t = block_sum(acc, sm);
  if (threadIdx.x == 0) {
    partial[blockIdx.x] = t;
    __threadfence();
    last = atomicAdd(counter, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (last) {
    __threadfence();
    double s = 0.0;
    for (unsigned b = threadIdx.x; b < gridDim.x; b += TPB) s += __ldcg(partial + b);
    const double tot = block_sum(s, sm);
    if (threadIdx.x == 0) {
      *out_nrm2 = tot;
      *counter = 0;
      if (ha.on) hess_update(ha.sp, ha.k, ha.rnorm_dev, ha.rnorm_host);
    }
  }
}

// y = a*x (+ b*z)   with a read from device memory as  a = *pa  (or 1/sqrt-free: the caller prepares it)
__global__ void scale_kernel2(double* __restrict__ y, const double* __restrict__ x, const double* __restrict__ pa, long long n) {
  pdl_go();
  pdl_wait();
  const double a = *pa;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) y[i] = a * x[i];
}

// r = b - w
__global__ void residual_kernel(double* __restrict__ r, const double* __restrict__ b, const double* __restrict__ w, long long n) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) r[i] = b[i] - w[i];
}

// beta^2 in scr[0]  ->  g = beta e_1, scr[1] = 1/beta, report beta
__global__ void init_cycle_kernel(SmallPtrs p, double* rnorm_dev, double* rnorm_host) {
  const double beta = sqrt(p.scr[0]);
  for (int i = 0; i <= p.m; i++) p.g[i] = 0.0;
  p.g[0] = beta;
  p.scr[1] = beta > 0.0 ? 1.0 / beta : 0.0;
  *rnorm_dev = beta;
  *rnorm_host = beta;
  __threadfence_system();
}

// Column k of the Hessenberg matrix: hcol[0..k] = V_j . w, hcol[k+1] = ||w||^2 after orthogonalisation.
__device__ void hess_update(const SmallPtrs& p, int k, double* rnorm_dev, double* rnorm_host) {
  const int ld = p.m + 1;
  double* col = p.H + (size_t)k * ld;
  const double hn = sqrt(p.hcol[k + 1]);
  for (int i = 0; i <= k; i++) col[i] = p.hcol[i];
  // previous rotations act on (col[i], col[i+1]), i < k; the sub-diagonal entry hn only meets the new one
  for (int i = 0; i < k; i++) {
    const double a = col[i], b = col[i + 1];
    col[i] = p.cs[i] * a + p.sn[i] * b;
    col[i + 1] = -p.sn[i] * a + p.cs[i] * b;
  }
  const double next = hn;
  // new rotation annihilating hn
  const double a = col[k];
  const double rr = sqrt(a * a + next * next);
  double c = 1.0, s = 0.0;
  if (rr > 0.0) {
    c = a / rr;
    s = next / rr;
  }
  p.cs[k] = c;
  p.sn[k] = s;
  col[k] = rr;
  const double gk = p.g[k];
  p.g[k] = c * gk;
  p.g[k + 1] = -s * gk;
  p.scr[1] = hn > 0.0 ? 1.0 / hn : 0.0;  // scaling of the next basis vector
  const double rn = fabs(p.g[k + 1]);
  *rnorm_dev = rn;
  *rnorm_host = rn;
  __threadfence_system();
}

__global__ void hess_kernel(SmallPtrs p, int k, double* rnorm_dev, double* rnorm_host) { hess_update(p, k, rnorm_dev, rnorm_host); }

// y = R^{-1} g for the first kk columns
__global__ void backsolve_kernel(SmallPtrs p, int kk) {
  const int ld = p.m + 1;
  for (int i = kk - 1; i >= 0; i--) {
    double t = p.g[i];
    for (int j = i + 1; j < kk; j++) t -= p.H[(size_t)j * ld + i] * p.y[j];
    const double d = p.H[(size_t)i * ld + i];
    p.y[i] = d != 0.0 ? t / d : 0.0;
  }
}

// Sum over the ranks of k <= 64 doubles through peer memory, in rank order (same bits on every rank).
struct SlotPtrs {
  double* s[SB200_MAX_RANKS];
};
__global__ void allreduce_kernel(SymmFlags sf, SlotPtrs sp, double* vals, int k, unsigned long long epoch) {
  const int t = threadIdx.x;
  const int par = (int)(epoch & 1);
  if (t < k) {
    const double v = vals[t];
    for (int q = 0; q < sf.nranks; q++) sp.s[q][((size_t)par * SB200_MAX_RANKS + sf.rank) * SLOT + t] = v;
  }
  __syncthreads();  // the block's stores happen-before thread 0's fence
  if (t == 0) {
    __threadfence_system();
    for (int q = 0; q < sf.nranks; q++) st_relaxed_sys(sf.f[q] + SYMM_AR + sf.rank, epoch);
  }
  if (t < sf.nranks) spin_until(sf.f[sf.rank] + SYMM_AR + t, epoch, sf.f[sf.rank]);
  __syncthreads();
  if (t < k) {
    double s = 0.0;
    const double* mine = sp.s[sf.rank];
    for (int q = 0; q < sf.nranks; q++) s += __ldcg(mine + ((size_t)par * SB200_MAX_RANKS + q) * SLOT + t);
    vals[t] = s;
  }
}

}  // namespace

int KspCtx::create(long long n, int restart, int rank, int nranks, KspCtx** out) {
  SB_CHECK(out, SB200_ERR_ARG, "null pointer");
  SB_CHECK(n >= 0 && restart >= 1 && restart <= 62, SB200_ERR_USER, "KSP: vector length must be >= 0 and 1 <= restart <= 62");
  KspCtx* k = new KspCtx();
  int rc = k->init(n, restart, rank, nranks);
  if (rc) {
    delete k;
    return rc;
  }
  *out = k;
  return 0;
}

int KspCtx::init(long long n_, int restart_, int rank, int nranks) {
  n = n_;
  restart = restart_;
  ldv = (n + 1) & ~1ll;  // even leading dimension: every basis vector starts 16-byte aligned
  if (ldv < 2) ldv = 2;
  const size_t nb = (size_t)ldv * sizeof(double);
  SB_CUDA(cudaMalloc((void**)&V, nb * (restart + 1)));
  // Z (the preconditioned vectors of the flexible variant) is allocated by the first solve that has a preconditioner: without one
  // the basis itself plays that role, and the inner solves of the saddle-point PCs never set one.  On a slab partition it is
  // allocated here: a solve is a collective there, and no rank may enter an allocating call while its peers' kernels wait for it.
  if (nranks > 1) SB_CUDA(cudaMalloc((void**)&Z, nb * restart));
  SB_CUDA(cudaMalloc((void**)&w, nb));
  SB_CUDA(cudaMalloc((void**)&small, SmallPtrs::count(restart) * sizeof(double)));
  SB_CUDA(cudaMemset(small, 0, SmallPtrs::count(restart) * sizeof(double)));
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int per_sm = 8;  // measured best (profiles/r02_notes.md)
  nblocks = (int)std::min<long long>((n + TPB - 1) / TPB > 0 ? (n + TPB - 1) / TPB : 1, (long long)sms * per_sm);
  SB_CUDA(cudaMalloc((void**)&partial, (size_t)nblocks * 64 * sizeof(double)));
  SB_CUDA(cudaMalloc((void**)&counters, 64 * sizeof(unsigned)));
  SB_CUDA(cudaMemset(counters, 0, 64 * sizeof(unsigned)));
  SB_CUDA(cudaHostAlloc((void**)&h_rnorm, 64, cudaHostAllocMapped));
  SB_CUDA(cudaHostGetDevicePointer((void**)&d_rnorm, h_rnorm, 0));
  for (auto& r : evr)
    for (auto& e : r) SB_CUDA(cudaEventCreate(&e));
  SB_TRY(arena.init(2 * SB200_MAX_RANKS * SLOT * sizeof(double), rank, nranks));
  SB_CHECK((slots = arena.alloc_doubles(2 * SB200_MAX_RANKS * SLOT)), SB200_ERR_CUDA, "arena exhausted");
  return 0;
}

KspCtx::~KspCtx() {
  if (V) cudaFree(V);
  if (Z) cudaFree(Z);
  if (w) cudaFree(w);
  if (small) cudaFree(small);
  if (partial) cudaFree(partial);
  if (counters) cudaFree(counters);
  if (h_rnorm) cudaFreeHost(h_rnorm);
  for (auto& r : evr)
    for (auto& e : r)
      if (e) cudaEventDestroy(e);
  arena.destroy();
}

int KspCtx::allreduce(double* vals, int k, cudaStream_t s) {
  if (arena.nranks == 1) return 0;
  SB_CHECK(arena.attached(), SB200_ERR_USER, "KSP on a slab partition: peers are not attached");
  SB_CHECK(k <= SLOT, SB200_ERR_USER, "all-reduce: too many values");
  SymmFlags sf;
  SlotPtrs sp;
  for (int q = 0; q < SB200_MAX_RANKS; q++) {
    sf.f[q] = q < arena.nranks ? arena.flags(q) : nullptr;
    sp.s[q] = q < arena.nranks ? arena.on(q, slots) : nullptr;
  }
  sf.rank = arena.rank;
  sf.nranks = arena.nranks;
  allreduce_kernel<<<1, 64, 0, s>>>(sf, sp, vals, k, ++ar_epoch);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return 0;
}

int KspCtx::dots(const double* x, const double* Y, long long ldy, int nv, double* out, cudaStream_t s) {
  const int vec2 = (reinterpret_cast<uintptr_t>(x) % 16 == 0 && reinterpret_cast<uintptr_t>(Y) % 16 == 0 && ldy % 2 == 0) ? 1 : 0;
  // 8 vectors per pass: measured on B200 (profiles/r02_notes.md) against 16 and 32 (registers, concurrent DRAM streams)
  SB_CUDA(launch_pdl(mdot_kernel<8>, dim3(nblocks, (nv + 7) / 8), dim3(TPB), s, x, Y, ldy, nv, n, partial, counters, out, vec2));
  count_launch();
  SB_CUDA(cudaGetLastError());
  return allreduce(out, nv, s);
}

int KspCtx::norm(const double* x, double* out, cudaStream_t s) { return dots(x, x, 0, 1, out, s); }

int KspCtx::solve(const double* b, double* x, bool guess_nonzero, cudaStream_t s) {
  SB_CHECK(op, SB200_ERR_USER, "KSP: no operator set (KSPSetOperators)");
  SB_CHECK(b && x && b != x, SB200_ERR_ARG, "KSPSolve: b and x must be distinct non-null vectors");
  const SmallPtrs sp = SmallPtrs::make(small, restart);
  const long long ld = ldv;
  auto al16 = [](const void* p) { return reinterpret_cast<uintptr_t>(p) % 16 == 0; };
  const int vx = al16(x) ? 1 : 0;  // V, Z, w are 256-byte aligned with an even leading dimension
  const int g1 = nblocks;
  its = 0;
  reason = 0;
  history.clear();
  t_op = t_pc = t_orth = 0.0;
  if (pc && !Z) SB_CUDA(cudaMalloc((void**)&Z, (size_t)ldv * sizeof(double) * restart));
  double* Zb = pc ? Z : V;  // without a PC the preconditioned vectors are the basis itself

  // ||b|| for KSPConvergedDefault
  SB_TRY(norm(b, sp.scr + 2, s));
  double b2 = 0.0;
  SB_CUDA(cudaMemcpyAsync(&b2, sp.scr + 2, sizeof(double), cudaMemcpyDeviceToHost, s));
  SB_CUDA(cudaStreamSynchronize(s));
  bnorm = std::sqrt(b2);
  if (!guess_nonzero) SB_CUDA(cudaMemsetAsync(x, 0, (size_t)n * sizeof(double), s));
  const double ttol = std::max(rtol * bnorm, atol);

  while (true) {
    // r = b - A x  -> V_0
    if (guess_nonzero || its > 0) {
      SB_TRY(op(op_ctx, x, w, (void*)s));
      residual_kernel<<<g1, TPB, 0, s>>>(V, b, w, n);
      count_launch();
    } else {
      SB_CUDA(cudaMemcpyAsync(V, b, (size_t)n * sizeof(double), cudaMemcpyDeviceToDevice, s));
    }
    SB_TRY(norm(V, sp.scr, s));
    init_cycle_kernel<<<1, 1, 0, s>>>(sp, sp.scr + 3, d_rnorm);
    count_launch();
    scale_kernel2<<<g1, TPB, 0, s>>>(V, V, sp.scr + 1, n);
    count_launch();
    SB_CUDA(cudaStreamSynchronize(s));
    rnorm = *h_rnorm;
    if (its == 0) history.push_back(rnorm);
    if (rnorm <= ttol) {
      reason = rnorm <= atol ? 3 : 2;  // KSP_CONVERGED_ATOL / RTOL
      return 0;
    }
    if (!(rnorm == rnorm)) {
      reason = -9;  // KSP_DIVERGED_NANORINF
      return 0;
    }
    // Arnoldi steps of this cycle.  lookahead = 0: one host read per iteration before the next one is enqueued (PETSc's decision
    // point).  lookahead = 1 (opt-in): iteration k+1 is enqueued before iteration k's norm is read, so the GPU never idles on the
    // host; when iteration k turns out to be the last, the speculative step behind it is discarded (it touches nothing the
    // back-substitution over k+1 columns reads) - at most one extra operator / preconditioner application per solve.
    int k_enq = 0, k = 0;  // enqueued / accounted iterations of this cycle
    bool done = false;
    auto enqueue = [&](int kq) -> int {
      double* vk = V + (size_t)kq * ld;
      double* zk = Zb + (size_t)kq * ld;
      cudaEvent_t* e = evr[kq % NRING];
      SB_CUDA(cudaEventRecord(e[0], s));
      if (pc) SB_TRY(pc(pc_ctx, vk, zk, (void*)s));
      SB_CUDA(cudaEventRecord(e[1], s));
      SB_TRY(op(op_ctx, zk, w, (void*)s));
      SB_CUDA(cudaEventRecord(e[2], s));
      SB_TRY(dots(w, V, ld, kq + 1, sp.hcol, s));  // classical Gram-Schmidt: all projections at once
      HessArgs ha;
      ha.sp = sp;
      ha.on = arena.nranks == 1 ? 1 : 0;  // single rank: the norm's last block also updates the Hessenberg column (one launch fewer)
      ha.k = kq;
      ha.rnorm_dev = sp.scr + 3;
      ha.rnorm_host = d_rnorm + (kq % NRING);
      SB_CUDA(launch_pdl(maxpy_kernel, dim3(g1), dim3(TPB), s, w, (const double*)V, ld, kq + 1, (const double*)sp.hcol, -1.0, n, partial, counters + 32,
                         sp.hcol + (kq + 1), 1, ha, 1));  // desc = 1: L2 reuse after the multi-dot
      count_launch();
      if (!ha.on) {
        SB_TRY(allreduce(sp.hcol + (kq + 1), 1, s));
        hess_kernel<<<1, 1, 0, s>>>(sp, kq, sp.scr + 3, d_rnorm + (kq % NRING));
        count_launch();
      }
      SB_CUDA(launch_pdl(scale_kernel2, dim3(g1), dim3(TPB), s, V + (size_t)(kq + 1) * ld, (const double*)w, (const double*)(sp.scr + 1), n));
      count_launch();
      SB_CUDA(cudaEventRecord(e[3], s));
      SB_CUDA(cudaGetLastError());
      return 0;
    };
    while (!done) {
      while (k_enq < restart && k_enq - k <= lookahead && its + (k_enq - k) < maxits) {
        SB_TRY(enqueue(k_enq));
        k_enq++;
      }
      if (k == k_enq) break;  // the cycle is complete
      cudaEvent_t* e = evr[k % NRING];
      SB_CUDA(cudaEventSynchronize(e[3]));  // the one host read per iteration (as in PETSc: the norm decides)
      float ms = 0.f;
      cudaEventElapsedTime(&ms, e[0], e[1]);
      t_pc += ms;
      cudaEventElapsedTime(&ms, e[1], e[2]);
      t_op += ms;
      cudaEventElapsedTime(&ms, e[2], e[3]);
      t_orth += ms;
      rnorm = reinterpret_cast<volatile double*>(h_rnorm)[k % NRING];
      k++;
      its++;
      history.push_back(rnorm);
      if (rnorm <= ttol) {
        reason = rnorm <= atol ? 3 : 2;
        done = true;
      } else if (!(rnorm == rnorm)) {
        reason = -9;
        done = true;
      } else if (rnorm >= dtol * bnorm) {
        reason = -4;  // KSP_DIVERGED_DTOL
        done = true;
      } else if (its >= maxits) {
        reason = -3;  // KSP_DIVERGED_ITS
        done = true;
      }
    }
    // x += Z y with R y = g
    backsolve_kernel<<<1, 1, 0, s>>>(sp, k);
    count_launch();
    HessArgs nohess = {};
    maxpy_kernel<<<g1, TPB, 0, s>>>(x, Zb, ld, k, sp.y, 1.0, n, partial, counters + 32, nullptr, vx, nohess, 0);
    count_launch();
    SB_CUDA(cudaGetLastError());
    if (done) break;
  }
  SB_CUDA(cudaStreamSynchronize(s));
  SB_CHECK(!arena.failed(), SB200_ERR_CUDA, "KSPSolve: a device-side flag wait (all-reduce / barrier over the slab ranks) timed out; the result is undefined");
  return 0;
}

}  // namespace sb200
