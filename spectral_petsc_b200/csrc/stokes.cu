// Stokes operator shells (stokes.C:499-758) on device-resident fp64 vectors, Dirichlet boundary
// (-boundary 0, the only configuration the reference documents as working, README:64-68).
//
// Layouts follow the reference: local velocity AoS [node][k] (stokes.C:651), local pressure [node],
// global vector AoS per interior node [v_0..v_{d-1}, p] (stokes.C:867-877).  The VecScatters are
// structured pad/crop index arithmetic; VecStrideGather/Scatter (stokes.C:585,613) are folded into
// the derivative kernel's element stride/offset; the VecAXPY accumulations are its epilogue.
#include "stokes.h"

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <vector>

#include "../../include/spectral_b200.h"
#include "common.cuh"
#include "deriv.h"

namespace sb200 {

namespace {

struct NodeInfo {
  bool interior;
  long long gid;  // interior ordinal (walk order)
  long long did;  // boundary ordinal (walk order)
};

__device__ __forceinline__ NodeInfo decode_node(const GridDesc& gd, long long idx) {
  // walk-order semantics of StokesSetupDomain (stokes.C:791-879) / BlockIt::normal (util.C:70-82); in a slab
  // view axis-0 indices are global (offset gd.i0 inside gd.n0g) and the ordinals are local to this rank
  long long rem = idx, cnt = -gd.goff;
  bool prefix_int = true, bdy = false;
  const bool small = gd.m < (1ll << 31);  // 32-bit divisions are several times cheaper than 64-bit ones
  for (int j = 0; j < gd.d; j++) {
    const long long s = gd.stride[j];
    const int il = small ? (int)((unsigned)rem / (unsigned)s) : (int)(rem / s);
    rem -= (long long)il * s;
    const int i = gd.gidx(j, il), ext = gd.gext(j);
    const bool b = (i == 0) || (i == ext - 1);
    if (prefix_int) {
      int c = i - 1;
      c = c < 0 ? 0 : (c > ext - 2 ? ext - 2 : c);
      cnt += (long long)c * gd.istride[j];
      if (b) prefix_int = false;
    }
    bdy |= b;
  }
  NodeInfo n;
  n.interior = !bdy;
  n.gid = cnt;
  n.did = idx - cnt;
  return n;
}

// local[node*nc + k] = interior ? src[gid*sstride + soff + k] : (dir ? dir[did*nc + k] : 0)
// Four nodes per thread and pass, all their loads issued before the first store (the kernel is latency bound otherwise).
template <int NC>
__global__ void pad_nodes_kernel(GridDesc gd, const double* __restrict__ src, int sstride, int soff,
                                 const double* __restrict__ dir, double* __restrict__ local) {
  constexpr int U = 4;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long idx0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx0 < gd.m; idx0 += U * stride) {
    double v[U][NC];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const long long idx = idx0 + u * stride;
      if (idx >= gd.m) continue;
      const NodeInfo n = decode_node(gd, idx);
#pragma unroll
      for (int k = 0; k < NC; k++) {
        if (n.interior) v[u][k] = src[n.gid * sstride + soff + k];
        else v[u][k] = dir ? dir[n.did * NC + k] : 0.0;
      }
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const long long idx = idx0 + u * stride;
      if (idx >= gd.m) continue;
#pragma unroll
      for (int k = 0; k < NC; k++) local[idx * NC + k] = v[u][k];
    }
  }
}

// dst[gid*dstride + doff + k] (=|+=) local[node*nc + k] (- sub[gid*dstride + doff + k]) at interior nodes
__global__ void crop_nodes_kernel(GridDesc gd, int nc, const double* __restrict__ local, double* __restrict__ dst,
                                  int dstride, int doff, int add, const double* __restrict__ sub) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < gd.m; idx += stride) {
    const NodeInfo n = decode_node(gd, idx);
    if (!n.interior) continue;
    for (int k = 0; k < nc; k++) {
      const long long e = n.gid * dstride + doff + k;
      double v = local[idx * nc + k];
      if (add) v = dst[e] + v;             // VecAXPY(vG1, 1.0, vG0) stokes.C:513,750
      if (sub) v = v + (-1.0) * sub[e];    // VecAXPY(yG, -1.0, force) stokes.C:756
      dst[e] = v;
    }
  }
}

struct TermPtrs {
  const double* t[3];
};

// dst[gid*dstride + doff + k] = ((0 +- T_0) +- T_1) +- T_2 at interior nodes: the VecAXPY chain of stokes.C:584-590 /
// 668-671 (w0 = 0; w0 -= D_i V_i in axis order) applied while cropping, same operation order as the reference.
// Two nodes per thread and pass, every load issued before the first use.
template <int NC, int NT>
__global__ void crop_sum_kernel(GridDesc gd, TermPtrs tp, double sign, double* __restrict__ dst, int dstride, int doff) {
  constexpr int U = 2;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long idx0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx0 < gd.m; idx0 += U * stride) {
    double v[U][NT][NC];
    NodeInfo nd[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const long long idx = idx0 + u * stride;
      nd[u].interior = false;
      if (idx >= gd.m) continue;
      nd[u] = decode_node(gd, idx);
      if (!nd[u].interior) continue;
#pragma unroll
      for (int t = 0; t < NT; t++)
#pragma unroll
        for (int k = 0; k < NC; k++) v[u][t][k] = tp.t[t][idx * NC + k];
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      if (!nd[u].interior) continue;
#pragma unroll
      for (int k = 0; k < NC; k++) {
        double a = 0.0;
#pragma unroll
        for (int t = 0; t < NT; t++) a = __dadd_rn(a, __dmul_rn(sign, v[u][t][k]));
        dst[nd[u].gid * dstride + doff + k] = a;
      }
    }
  }
}

// dst[gid*dstride + doff] = ((0 + G_0[node*d + 0]) + G_1[node*d + 1]) + G_2[node*d + 2] at interior nodes, G_i = D_i v (m*d each):
// the divergence as the trace of the velocity gradient, accumulated in the order of stokes.C:584-590 with the arithmetic of
// crop_sum_kernel(sign = 1), so the result has the bits of the separate StokesDivergence pass.
__global__ void crop_trace_kernel(GridDesc gd, int d, TermPtrs tp, double* __restrict__ dst, int dstride, int doff) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < gd.m; idx += stride) {
    const NodeInfo n = decode_node(gd, idx);
    if (!n.interior) continue;
    double v = 0.0;
    for (int t = 0; t < d; t++) v = __dadd_rn(v, __dmul_rn(1.0, tp.t[t][idx * d + t]));
    dst[n.gid * dstride + doff] = v;
  }
}

template <int D>
struct VPtrs {
  double* v[D];
  const double* s[D];
};

// stokes.C:647-662: symmetrise, z = eps:E0, v = eta*eps + deta*E0*z
// FOLD (opt-in, StokesCtx::fold_pressure): v_jj -= pl, the boundary-extrapolated local pressure, so that the viscous tail
// -sum_j D_j V_j also produces the pressure gradient D_i p of StokesMatMultVP (stokes.C:611-614).  FOLD = false compiles to the
// kernel as it was.
// Fused divergence rows (StokesCtx::trace_divergence): div[gid*div_stride + div_off] = ((0 + g_00) + g_11) + g_22 at interior nodes,
// the arithmetic of crop_trace_kernel, taken from the gradient in registers before the flux overwrites it.
struct DivDst {
  double* dst;
  int stride, off;
};

template <int D, bool FOLD = false>
__global__ void vv_flux_kernel(long long m, const double* __restrict__ eta, const double* __restrict__ deta, VPtrs<D> p,
                               const double* __restrict__ pl, GridDesc gd, DivDst dv) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += stride) {
    double g[D][D], st[D][D], S0[D][D];
#pragma unroll
    for (int j = 0; j < D; j++)
#pragma unroll
      for (int k = 0; k < D; k++) {
        g[j][k] = p.v[j][i * D + k];
        S0[j][k] = p.s[j][i * D + k];
      }
    if (dv.dst) {
      const NodeInfo nd = decode_node(gd, i);
      if (nd.interior) {
        double tr = 0.0;
#pragma unroll
        for (int j = 0; j < D; j++) tr = __dadd_rn(tr, __dmul_rn(1.0, g[j][j]));
        dv.dst[nd.gid * dv.stride + dv.off] = tr;
      }
    }
    double z = 0.0;
#pragma unroll
    for (int j = 0; j < D; j++)
#pragma unroll
      for (int k = 0; k < D; k++) {
        st[j][k] = __dmul_rn(0.5, __dadd_rn(g[j][k], g[k][j]));
        z = __dadd_rn(z, __dmul_rn(st[j][k], S0[j][k]));
      }
    const double e = eta[i], de = deta[i];
    const double pli = FOLD ? pl[i] : 0.0;
#pragma unroll
    for (int j = 0; j < D; j++)
#pragma unroll
      for (int k = 0; k < D; k++) {
        const double s = __dmul_rn(e, st[j][k]);
        double val = __dadd_rn(s, __dmul_rn(__dmul_rn(de, S0[j][k]), z));
        if (FOLD && j == k) val = __dadd_rn(val, -pli);
        p.v[j][i * D + k] = val;
      }
  }
}

struct Rheo {
  int type;
  double hardness, exponent, regularization, gamma0;
};

__device__ __forceinline__ double atomicMinD(double* addr, double v) {
  unsigned long long* a = (unsigned long long*)addr;
  unsigned long long old = *a, assumed;
  do {
    assumed = old;
    if (__longlong_as_double(assumed) <= v) break;
    old = atomicCAS(a, assumed, __double_as_longlong(v));
  } while (assumed != old);
  return __longlong_as_double(old);
}
__device__ __forceinline__ double atomicMaxD(double* addr, double v) {
  unsigned long long* a = (unsigned long long*)addr;
  unsigned long long old = *a, assumed;
  do {
    assumed = old;
    if (__longlong_as_double(assumed) >= v) break;
    old = atomicCAS(a, assumed, __double_as_longlong(v));
  } while (assumed != old);
  return __longlong_as_double(old);
}

// stokes.C:708-725 + rheology (stokes.C:1920-1944): s = sym(grad v), gamma = 1/2 s:s, eta/deta, V = eta*s, strain = s
template <int D, bool FOLD = false>
__global__ void rheology_kernel(long long m, Rheo r, double* __restrict__ eta, double* __restrict__ deta, VPtrs<D> p,
                                double* __restrict__ minmax, const double* __restrict__ pl, GridDesc gd, DivDst dv) {
  // p.s[j] (const view) and the written strain are the same arrays: strain is read raw and overwritten
  const long long stride = (long long)gridDim.x * blockDim.x;
  double lmin = DBL_MAX, lmax = -DBL_MAX;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += stride) {
    double g[D][D], s[D][D];
#pragma unroll
    for (int j = 0; j < D; j++)
#pragma unroll
      for (int k = 0; k < D; k++) g[j][k] = p.s[j][i * D + k];
    if (dv.dst) {
      const NodeInfo nd = decode_node(gd, i);
      if (nd.interior) {
        double tr = 0.0;
#pragma unroll
        for (int j = 0; j < D; j++) tr = __dadd_rn(tr, __dmul_rn(1.0, g[j][j]));
        dv.dst[nd.gid * dv.stride + dv.off] = tr;
      }
    }
    double gamma = 0.0;
#pragma unroll
    for (int j = 0; j < D; j++)
#pragma unroll
      for (int k = 0; k < D; k++) {
        s[j][k] = __dmul_rn(0.5, __dadd_rn(g[j][k], g[k][j]));
        gamma = __dadd_rn(gamma, __dmul_rn(0.5, __dmul_rn(s[j][k], s[j][k])));
      }
    double e, de;
    if (r.type == 0) {
      e = 1.0;
      de = 0.0;
    } else {
      const double n = r.exponent;
      const double pw = (1.0 - n) / (2.0 * n);
      const double base = __dadd_rn(r.regularization, gamma / r.gamma0);
      e = __dmul_rn(r.hardness, pow(base, pw));
      de = (fabs(n) > 1.0e-5) ? __dmul_rn(r.hardness * pw / r.gamma0, pow(base, pw - 1.0)) : 0.0;
    }
    eta[i] = e;
    deta[i] = de;
    lmin = fmin(lmin, e);
    lmax = fmax(lmax, e);
    double* sw[D];
#pragma unroll
    for (int j = 0; j < D; j++) sw[j] = const_cast<double*>(p.s[j]);
#pragma unroll
    for (int j = 0; j < D; j++)
#pragma unroll
      for (int k = 0; k < D; k++) {
        double val = __dmul_rn(e, s[j][k]);
        if (FOLD && j == k) val = __dadd_rn(val, -pl[i]);  // opt-in: V = eta*eps - p I, see vv_flux_kernel
        p.v[j][i * D + k] = val;
        sw[j][i * D + k] = s[j][k];
      }
  }
  // block reduce min/max (VecMin / VecMax, stokes.C:731-734) without a host sync
  for (int o = 16; o > 0; o >>= 1) {
    lmin = fmin(lmin, __shfl_xor_sync(0xffffffffu, lmin, o));
    lmax = fmax(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
  }
  if ((threadIdx.x & 31) == 0 && lmin <= lmax) {
    atomicMinD(minmax, lmin);
    atomicMaxD(minmax + 1, lmax);
  }
}

__global__ void init_minmax_kernel(double* mm) {
  mm[0] = DBL_MAX;
  mm[1] = -DBL_MAX;
}

__global__ void recip_crop_kernel(GridDesc gd, const double* __restrict__ eta, double* __restrict__ y) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < gd.m; idx += stride) {
    const NodeInfo n = decode_node(gd, idx);
    if (n.interior) y[n.gid] = 1.0 / eta[idx];  // scatterLP + VecReciprocal, stokes.C:549-551
  }
}

__global__ void scale_kernel(long long n, double a, double* __restrict__ y) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) y[i] = a * y[i];
}

// One pass of StokesPressureReduceOrder (stokes.C:1042-1074): along `axis`, set both end nodes of every
// selected line to the degree-(P-3) extrapolation of its interior values.  Lines are enumerated over
// the other axes; lo[j]/hi[j] bound the other indices (inclusive) so the three ordered passes touch
// exactly the nodes the reference's loops leave in the final array.
struct ReduceArgs {
  int axis;
  int lo[3], hi[3];
  long long stride[3];
  int P;
  int nother;       // number of other axes (d-1)
  int oax[2];       // the other axes, slowest first
  long long nlines;
};

__global__ void reduce_order_kernel(ReduceArgs a, const double* __restrict__ w0, const double* __restrict__ w1,
                                    double* __restrict__ pres) {
  // block = 32 lines (threadIdx.x, adjacent in memory) x 8 slices of the line (threadIdx.y): the loads of a warp
  // are coalesced across lines and every line's sum is finished through shared memory
  __shared__ double s0[8][33], s1[8][33];
  const long long line = (long long)blockIdx.x * 32 + threadIdx.x;
  const bool live = line < a.nlines;
  long long rem = live ? line : 0, base = 0;
  for (int q = a.nother - 1; q >= 0; q--) {
    const int ax = a.oax[q];
    const int ext = a.hi[ax] - a.lo[ax] + 1;
    const int i = a.lo[ax] + (int)(rem % ext);
    rem /= ext;
    base += (long long)i * a.stride[ax];
  }
  const long long s = a.stride[a.axis];
  double f0 = 0.0, f1 = 0.0;
  if (live)
    for (int k = 1 + threadIdx.y; k < a.P - 1; k += 8) {
      const double v = pres[base + k * s];
      f0 = fma(w0[k], v, f0);
      f1 = fma(w1[k], v, f1);
    }
  s0[threadIdx.y][threadIdx.x] = f0;
  s1[threadIdx.y][threadIdx.x] = f1;
  __syncthreads();
  if (threadIdx.y == 0 && live) {
    double t0 = 0.0, t1 = 0.0;
    for (int j = 0; j < 8; j++) {
      t0 += s0[j][threadIdx.x];
      t1 += s1[j][threadIdx.x];
    }
    pres[base] = t0;
    pres[base + (long long)(a.P - 1) * s] = t1;
  }
}

// Same pass for the LAST axis (contiguous lines): one warp per line, coalesced loads, shuffle reduction.
__global__ void reduce_order_lastaxis_kernel(ReduceArgs a, const double* __restrict__ w0, const double* __restrict__ w1,
                                             double* __restrict__ pres) {
  const long long line = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (line >= a.nlines) return;
  long long rem = line, base = 0;
  for (int q = a.nother - 1; q >= 0; q--) {
    const int ax = a.oax[q];
    const int ext = a.hi[ax] - a.lo[ax] + 1;
    const int i = a.lo[ax] + (int)(rem % ext);
    rem /= ext;
    base += (long long)i * a.stride[ax];
  }
  double f0 = 0.0, f1 = 0.0;
  for (int k = 1 + lane; k < a.P - 1; k += 32) {
    const double v = pres[base + k];
    f0 = fma(w0[k], v, f0);
    f1 = fma(w1[k], v, f1);
  }
  for (int o = 16; o > 0; o >>= 1) {
    f0 += __shfl_xor_sync(0xffffffffu, f0, o);
    f1 += __shfl_xor_sync(0xffffffffu, f1, o);
  }
  if (lane == 0) {
    pres[base] = f0;
    pres[base + (a.P - 1)] = f1;
  }
}

// The pressure pad (VecScatter global -> local, stokes.C:606-608) and the LAST-axis pass of the extrapolation in one kernel (single
// GPU): one warp per interior line reads the line's interior values from the global vector, forms the two end-point sums with the
// arithmetic of reduce_order_lastaxis_kernel (lane-strided fma chains, xor-shuffle tree) and writes the complete padded line.
// Lines on the boundary of another axis are left alone: the later passes write every one of their nodes before anything reads them.
__global__ void pad_reduce_lastaxis_kernel(GridDesc gd, const double* __restrict__ src, int sstride, int soff, const double* __restrict__ w0,
                                           const double* __restrict__ w1, double* __restrict__ pres) {
  const long long line = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int d = gd.d, P = gd.dim[d - 1];
  if (line >= gd.m / P) return;
  long long rem = line, gbase = -gd.goff;  // slab view: axis-0 indices are global, ordinals local to this rank
  bool inter = true;
  for (int j = d - 2; j >= 0; j--) {
    const int dj = gd.dim[j];
    const int il = (int)(rem % dj);
    rem /= dj;
    const int ij = gd.gidx(j, il), ext = gd.gext(j);
    inter = inter && ij >= 1 && ij <= ext - 2;
    gbase += (long long)(ij - 1) * gd.istride[j];
  }
  if (!inter) return;
  const double* __restrict__ sl = src + gbase * sstride + soff;  // interior node k (1 <= k <= P-2) at sl[(k-1)*sstride]
  double* __restrict__ pl = pres + line * P;
  double f0 = 0.0, f1 = 0.0;
  for (int k = 1 + lane; k < P - 1; k += 32) {
    const double v = sl[(long long)(k - 1) * sstride];
    pl[k] = v;
    f0 = fma(w0[k], v, f0);
    f1 = fma(w1[k], v, f1);
  }
  for (int o = 16; o > 0; o >>= 1) {
    f0 += __shfl_xor_sync(0xffffffffu, f0, o);
    f1 += __shfl_xor_sync(0xffffffffu, f1, o);
  }
  if (lane == 0) {
    pl[0] = f0;
    pl[P - 1] = f1;
  }
}

// Slab partition, extrapolation along the partitioned axis 0: every rank forms the two end-point sums over ITS
// planes for each of the R0 lines and pushes them to the owners of plane 0 (rank 0) and plane P-1 (last rank).
__global__ void reduce0_partial_kernel(const double* __restrict__ w0, const double* __restrict__ w1, const double* __restrict__ pres,
                                       int i0, int nloc, int P, long long R0, double* __restrict__ red_first, double* __restrict__ red_last) {
  const long long line = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (line >= R0) return;
  double f0 = 0.0, f1 = 0.0;
  for (int kl = 0; kl < nloc; kl++) {
    const int k = i0 + kl;
    if (k < 1 || k > P - 2) continue;
    const double v = pres[(long long)kl * R0 + line];
    f0 = fma(w0[k], v, f0);
    f1 = fma(w1[k], v, f1);
  }
  red_first[line] = f0;       // slot [rank][0][line] on rank 0
  red_last[R0 + line] = f1;   // slot [rank][1][line] on the last rank
}

__global__ void reduce0_finish_kernel(const double* __restrict__ red, int nranks, int which, long long R0, double* __restrict__ plane) {
  const long long line = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (line >= R0) return;
  double f = 0.0;
  for (int q = 0; q < nranks; q++) f += __ldcg(red + ((long long)q * 2 + which) * R0 + line);  // rank order: same on every run
  plane[line] = f;
}

int grid_for(long long n) {
  long long b = (n + 255) / 256;
  return (int)std::min<long long>(std::max<long long>(b, 1), 148 * 16);
}

// Lagrange weights l_k(x_end) on the interior CGL nodes x_1..x_{P-2}, in long double.
void extrap_weights(int P, std::vector<double>& w0, std::vector<double>& w1) {
  const long double pi = 3.14159265358979323846264338327950288L;
  std::vector<long double> x(P);
  for (int i = 0; i < P; i++) x[i] = cosl(pi * i / (P - 1));
  w0.assign(P, 0.0);
  w1.assign(P, 0.0);
  for (int k = 1; k < P - 1; k++) {
    long double a = 1.0L, b = 1.0L;
    for (int j = 1; j < P - 1; j++) {
      if (j == k) continue;
      a *= (x[0] - x[j]) / (x[k] - x[j]);
      b *= (x[P - 1] - x[j]) / (x[k] - x[j]);
    }
    w0[k] = (double)a;
    w1[k] = (double)b;
  }
}

}  // namespace

// ---- StokesCtx ---------------------------------------------------------------------------
int StokesCtx::create(int d, const int* dim, int rank, int nranks, StokesCtx** out) {
  SB_CHECK(d == 2 || d == 3, SB200_ERR_SUP, "Stokes shells are implemented for dimension 2 and 3 (stokes.C:1036)");
  StokesCtx* c = new StokesCtx();
  int rc = c->init(d, dim, rank, nranks);
  if (rc) {
    delete c;
    return rc;
  }
  *out = c;
  return 0;
}

int StokesCtx::init(int d, const int* dim, int rank, int nranks) {
  SB_TRY(gd.init_slab(d, dim, rank, nranks));
  for (int k = 0; k < d; k++) gdim[k] = dim[k];
  gp = gd.g;
  gv = gd.g * d;
  g = gd.g * (d + 1);
  dvn = (gd.m - gd.g) * d;
  const size_t mb = (size_t)gd.m * sizeof(double);
  const size_t lines0 = (size_t)gd.stride[0];
  // one peer-mapped arena, same allocation order on every rank
  const size_t total = (size_t)(3 + d + (nranks > 1 ? 2 : 0)) * (mb * d + 256) + 3 * (mb + 256) + (size_t)d * (mb * d + 256) + 2 * (mb + 256) +
                       ((size_t)nranks * 2 * lines0 * sizeof(double) + 256);
  SB_TRY(arena.init(total, rank, nranks));
  for (int k = 0; k < 3 + d; k++) SB_CHECK((workV[k] = arena.alloc_doubles((size_t)gd.m * d)), SB200_ERR_CUDA, "arena exhausted");  // xL, yL, V[d], term
  for (int k = 0; k < 3; k++) SB_CHECK((workP[k] = arena.alloc_doubles(gd.m)), SB200_ERR_CUDA, "arena exhausted");
  for (int k = 0; k < d; k++) {
    SB_CHECK((strain[k] = arena.alloc_doubles((size_t)gd.m * d)), SB200_ERR_CUDA, "arena exhausted");
    SB_CUDA(cudaMemset(strain[k], 0, mb * d));
  }
  SB_CHECK((eta = arena.alloc_doubles(gd.m)), SB200_ERR_CUDA, "arena exhausted");
  SB_CHECK((deta = arena.alloc_doubles(gd.m)), SB200_ERR_CUDA, "arena exhausted");
  SB_CHECK((red = arena.alloc_doubles((size_t)nranks * 2 * lines0)), SB200_ERR_CUDA, "arena exhausted");
  if (nranks > 1) {
    SB_CHECK((Xp = arena.alloc_doubles((size_t)gd.m * d)), SB200_ERR_CUDA, "arena exhausted");
    SB_CHECK((Yp = arena.alloc_doubles((size_t)gd.m * d)), SB200_ERR_CUDA, "arena exhausted");
  }
  {
    std::vector<double> ones((size_t)gd.m, 1.0);
    SB_CUDA(cudaMemcpy(eta, ones.data(), mb, cudaMemcpyHostToDevice));
    SB_CUDA(cudaMemset(deta, 0, mb));
  }
  SB_CUDA(cudaMalloc((void**)&dirichlet, std::max<size_t>(8, (size_t)dvn * sizeof(double))));
  SB_CUDA(cudaMemset(dirichlet, 0, std::max<size_t>(8, (size_t)dvn * sizeof(double))));
  SB_CUDA(cudaMalloc((void**)&force, std::max<size_t>(8, (size_t)g * sizeof(double))));
  SB_CUDA(cudaMemset(force, 0, std::max<size_t>(8, (size_t)g * sizeof(double))));
  SB_CUDA(cudaMalloc((void**)&vG0, std::max<size_t>(8, (size_t)gv * sizeof(double))));
  SB_CUDA(cudaMalloc((void**)&vG1, std::max<size_t>(8, (size_t)gv * sizeof(double))));
  SB_CUDA(cudaMalloc((void**)&minmax, 2 * sizeof(double)));
  SB_CUDA(cudaMalloc((void**)&sync, 64));
  // side stream: on a slab partition the local-axis derivative batch runs there beside the axis-0 pencil chain; on one GPU the pressure
  // pad + boundary extrapolation (small latency-bound kernels) run there beside the velocity pad and the gradient batch
  SB_CUDA(cudaStreamCreateWithFlags(&aux_stream, cudaStreamNonBlocking));
  SB_CUDA(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
  SB_CUDA(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
  SB_CUDA(cudaEventCreateWithFlags(&ev_pjoin, cudaEventDisableTiming));
  SB_CUDA(cudaMemset(sync, 0, 64));
  for (int k = 0; k < d; k++) {
    Dax[k] = nullptr;
    for (int q = 0; q < k; q++)
      if (gdim[q] == gdim[k]) {
        Dax[k] = Dax[q];
        w0[k] = w0[q];
        w1[k] = w1[q];
      }
    if (!Dax[k]) {
      DiffMatrix* dm = new DiffMatrix();
      SB_TRY(DiffMatrix::create(gdim[k], dm));
      owned.push_back(dm);
      Dax[k] = dm;
      std::vector<double> a, b;
      extrap_weights(gdim[k], a, b);
      SB_CUDA(cudaMalloc((void**)&w0[k], a.size() * sizeof(double)));
      SB_CUDA(cudaMalloc((void**)&w1[k], b.size() * sizeof(double)));
      SB_CUDA(cudaMemcpy(w0[k], a.data(), a.size() * sizeof(double), cudaMemcpyHostToDevice));
      SB_CUDA(cudaMemcpy(w1[k], b.data(), b.size() * sizeof(double), cudaMemcpyHostToDevice));
      owned_w.push_back(w0[k]);
      owned_w.push_back(w1[k]);
    }
  }
  return 0;
}

StokesCtx::~StokesCtx() {
  if (aux_stream) {
    cudaStreamSynchronize(aux_stream);
    cudaStreamDestroy(aux_stream);
  }
  if (ev_fork) cudaEventDestroy(ev_fork);
  if (ev_join) cudaEventDestroy(ev_join);
  if (ev_pjoin) cudaEventDestroy(ev_pjoin);
  arena.destroy();
  if (dirichlet) cudaFree(dirichlet);
  if (force) cudaFree(force);
  if (vG0) cudaFree(vG0);
  if (vG1) cudaFree(vG1);
  if (minmax) cudaFree(minmax);
  if (sync) cudaFree(sync);
  for (double* p : owned_w) cudaFree(p);
  for (DiffMatrix* dm : owned) {
    dm->destroy();
    delete dm;
  }
}

// Launch one derivative; along the partitioned axis the operand rows are pulled from the planes' owners
// (x must be an arena array), bracketed by device-side barriers (see EllipticCtx::deriv).
int StokesCtx::deriv_common(DerivParams& p, int axis, cudaStream_t s) {
  if (axis == 0 && arena.nranks > 1) {
    SB_CHECK(arena.attached(), SB200_ERR_USER, "slab partition: peers are not attached (exchange the IPC handles first)");
    if (slab_deriv0_pencil_supported(arena, p)) return slab_deriv0_pencil(arena, p, gd.dim[0], gd.i0, Xp, Yp, s);
    p.npeer = arena.nranks;
    p.nloc = gd.dim[0];
    p.row0 = gd.i0;
    for (int q = 0; q < arena.nranks; q++) p.xpeer[q] = arena.on(q, p.x);
    SB_TRY(arena.barrier(s));
    SB_TRY(deriv_apply(p, s));
    return arena.barrier(s);
  }
  return deriv_apply(p, s);
}

DerivParams StokesCtx::job_v(int axis, const double* x, double* y, const double* yin, int mode) const {
  // DV[axis]: rank d+1 with trailing component axis of extent d (stokes.C:284-289)
  DerivParams p;
  p.D = Dax[axis]->d_D;
  p.Ae = Dax[axis]->d_Aep;
  p.Bo = Dax[axis]->d_Bop;
  p.HP = Dax[axis]->HP;
  p.sync = sync;
  p.P = Dax[axis]->P;
  p.Pp = Dax[axis]->Pp;
  p.x = x;
  p.y = y;
  p.yin = yin;
  p.O = gd.m / (gd.stride[axis] * gd.dim[axis]);
  p.R = gd.stride[axis] * gd.d;
  p.xs = p.ys = 1;
  p.xoff = p.yoff = 0;
  p.mode = mode;
  return p;
}

DerivParams StokesCtx::job_p(int axis, const double* x, int xs, int xoff, double* y, int ys, int yoff, const double* yin,
                             int mode) const {
  // DP[axis] on a scalar field that may live inside an AoS vector (VecStrideGather/Scatter, stokes.C:585,613)
  DerivParams p;
  p.D = Dax[axis]->d_D;
  p.Ae = Dax[axis]->d_Aep;
  p.Bo = Dax[axis]->d_Bop;
  p.HP = Dax[axis]->HP;
  p.sync = sync;
  p.P = Dax[axis]->P;
  p.Pp = Dax[axis]->Pp;
  p.x = x;
  p.y = y;
  p.yin = yin;
  p.O = gd.m / (gd.stride[axis] * gd.dim[axis]);
  p.R = gd.stride[axis];
  p.xs = xs;
  p.xoff = xoff;
  p.ys = ys;
  p.yoff = yoff;
  p.mode = mode;
  return p;
}

int StokesCtx::deriv_v(int axis, const double* x, double* y, const double* yin, int mode, cudaStream_t s) {
  DerivParams p = job_v(axis, x, y, yin, mode);
  return deriv_common(p, axis, s);
}

int StokesCtx::deriv_p(int axis, const double* x, int xs, int xoff, double* y, int ys, int yoff, const double* yin,
                       int mode, cudaStream_t s) {
  DerivParams p = job_p(axis, x, xs, xoff, y, ys, yoff, yin, mode);
  return deriv_common(p, axis, s);
}

bool StokesCtx::batchable() const {
  if (gd.d > SB200_EO_MAX_JOBS) return false;
  if (arena.nranks > 1 && gd.stride[0] % arena.nranks != 0) return false;  // the axis-0 pencils need R0 % G == 0
  for (int k = 1; k < gd.d; k++)
    if (Dax[k] != Dax[0]) return false;
  DerivParams p = job_p(0, workP[0], 1, 0, workP[1], 1, 0, nullptr, DERIV_STORE);
  return deriv_eo_supported(p);
}

// Single GPU, every axis within the even-odd kernel's reach (P <= SB200_EO_MAX_P): the scatters and AXPY chains around the
// derivatives run inside the derivative launches (fused pad loader, fused crop-sum epilogue; deriv.h), whatever the extents.
bool StokesCtx::fusable() const {
  if (arena.nranks > 1) return false;
  for (int k = 0; k < gd.d; k++) {
    DerivParams p = job_p(k, workP[0], 1, 0, workP[1], 1, 0, nullptr, DERIV_STORE);
    if (!deriv_eo_supported(p)) return false;
  }
  return true;
}

EoLineMap StokesCtx::line_map(int axis, int nc) const {
  EoLineMap lm;
  lm.d = gd.d;
  lm.nc = nc;
  lm.axis = axis;
  for (int j = 0; j < gd.d; j++) {
    lm.dim[j] = gd.dim[j];
    lm.istride[j] = gd.istride[j];
  }
  return lm;
}

// The d independent derivatives of one stage.  Single GPU: one batched even-odd launch when the axes share the matrix (equal
// extents), else one launch per axis in order (a job's terms then come from earlier launches).  Slab: axis 0 goes through the
// pencils (two pushes over NVLink), the local axes run as one batch.
int StokesCtx::run_jobs(DerivParams* jobs, int d, cudaStream_t s) {
  if (arena.nranks == 1) return deriv_eo_jobs(jobs, d, sync, s);
  if (!slab_deriv0_pencil_supported(arena, jobs[0])) {
    SB_TRY(deriv_common(jobs[0], 0, s));
    if (d > 1) SB_TRY(deriv_eo_batch(jobs + 1, d - 1, sync, s));
    return 0;
  }
  // The axis-0 chain (push the operand planes into the pencils, barrier, differentiate the pencil, push the rows back, barrier) runs on
  // the caller's stream; the local axes run CONCURRENTLY on the context's side stream (their own ticket counters): the two pushes and the
  // two cross-GPU barriers no longer sit in front of / behind 40 us of local work (profiles/r02_stokes_slab_profile_n2.txt).
  if (d > 1) {
    SB_CUDA(cudaEventRecord(ev_fork, s));
    SB_CUDA(cudaStreamWaitEvent(aux_stream, ev_fork, 0));
    SB_TRY(deriv_eo_batch(jobs + 1, d - 1, sync + 4, aux_stream));
    SB_CUDA(cudaEventRecord(ev_join, aux_stream));
  }
  SB_TRY(slab_deriv0_pencil(arena, jobs[0], gd.dim[0], gd.i0, Xp, Yp, s));
  if (d > 1) SB_CUDA(cudaStreamWaitEvent(s, ev_join, 0));
  return 0;
}

int StokesCtx::crop_sum(int nc, int nterms, double* const* terms, double sign, double* dst, int dstride, int doff, cudaStream_t s) {
  TermPtrs tp;
  for (int t = 0; t < 3; t++) tp.t[t] = t < nterms ? terms[t] : nullptr;
  const int g = grid_for(gd.m);
  if (nc == 3 && nterms == 3) crop_sum_kernel<3, 3><<<g, 256, 0, s>>>(gd, tp, sign, dst, dstride, doff);
  else if (nc == 1 && nterms == 3) crop_sum_kernel<1, 3><<<g, 256, 0, s>>>(gd, tp, sign, dst, dstride, doff);
  else if (nc == 2 && nterms == 2) crop_sum_kernel<2, 2><<<g, 256, 0, s>>>(gd, tp, sign, dst, dstride, doff);
  else if (nc == 1 && nterms == 2) crop_sum_kernel<1, 2><<<g, 256, 0, s>>>(gd, tp, sign, dst, dstride, doff);
  else {
    set_last_error("crop_sum: unsupported component / term count");
    return SB200_ERR_SUP;
  }
  count_launch();
  SB_CUDA(cudaGetLastError());
  return 0;
}

int StokesCtx::crop_trace(double* const* grads, double* dst, int dstride, int doff, cudaStream_t s) {
  TermPtrs tp;
  for (int t = 0; t < 3; t++) tp.t[t] = t < gd.d ? grads[t] : nullptr;
  crop_trace_kernel<<<grid_for(gd.m), 256, 0, s>>>(gd, gd.d, tp, dst, dstride, doff);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return 0;
}

int StokesCtx::pad_vel(const double* src, int sstride, int soff, bool with_dirichlet, double* local, cudaStream_t s) {
  if (gd.d == 2) pad_nodes_kernel<2><<<grid_for(gd.m), 256, 0, s>>>(gd, src, sstride, soff, with_dirichlet ? dirichlet : nullptr, local);
  else pad_nodes_kernel<3><<<grid_for(gd.m), 256, 0, s>>>(gd, src, sstride, soff, with_dirichlet ? dirichlet : nullptr, local);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return 0;
}

int StokesCtx::pad_pres(const double* src, int sstride, int soff, double* local, cudaStream_t s) {
  pad_nodes_kernel<1><<<grid_for(gd.m), 256, 0, s>>>(gd, src, sstride, soff, nullptr, local);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return 0;
}

int StokesCtx::crop(int nc, const double* local, double* dst, int dstride, int doff, bool add, const double* sub, cudaStream_t s) {
  crop_nodes_kernel<<<grid_for(gd.m), 256, 0, s>>>(gd, nc, local, dst, dstride, doff, add ? 1 : 0, sub);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return 0;
}

// y_vel[interior] (=|+=) -sum_j D_j V_j   with V from the pointwise step; shared tail of VV and Function
int StokesCtx::viscous_tail(double* dst, int dstride, int doff, cudaStream_t s) {
  const int d = gd.d;
  if (fusable() && gd.m <= SB200_FUSE_CROP_MAX_NODES) {
    // one launch: axes 1..d-1 store their terms D_i V_i, then axis 0 - whose 8-line blocks are contiguous in the AoS fields, so its
    // epilogue reads the terms with 16-byte loads - applies the "-=" chain (stokes.C:668-671) in AXIS order, its own value first,
    // and scatters into the global vector (:673): the arithmetic of crop_sum_kernel, no separate crop pass
    double* terms[2] = {workV[0], workV[1]};
    DerivParams jobs[3];
    for (int i = 1; i < d; i++) jobs[i - 1] = job_v(i, workV[2 + i], terms[i - 1], nullptr, DERIV_STORE);
    DerivParams& f = jobs[d - 1] = job_v(0, workV[2], nullptr, nullptr, DERIV_STORE);
    f.lm = line_map(0, d);
    f.gdst = dst;
    f.gd_stride = dstride;
    f.gd_off = doff;
    f.fin = EO_FIN_SUM;
    f.nterms = d - 1;
    f.self_pos = 0;
    for (int i = 0; i < d - 1; i++) f.term[i] = terms[i];
    f.sign = -1.0;
    return run_jobs(jobs, d, s);
  }
  if (fusable() || batchable()) {
    // one launch for the d terms D_i V_i, the "-=" chain (stokes.C:668-671) is applied by the crop in axis order
    double* terms[3] = {workV[0], workV[1], workV[2 + d]};
    DerivParams jobs[3];
    for (int i = 0; i < d; i++) jobs[i] = job_v(i, workV[2 + i], terms[i], nullptr, DERIV_STORE);
    SB_TRY(run_jobs(jobs, d, s));
    return crop_sum(d, d, terms, -1.0, dst, dstride, doff, s);
  }
  double* yL = workV[1];
  for (int i = 0; i < d; i++) SB_TRY(deriv_v(i, workV[2 + i], yL, i == 0 ? nullptr : yL, DERIV_SUB, s));  // :668-671
  return crop(d, yL, dst, dstride, doff, false, nullptr, s);
}

int StokesCtx::matmult_vv_into(const double* x, int xstride, int xoff, double* dst, int dstride, int doff, cudaStream_t s,
                               double* div_dst, int div_stride, int div_off, const double* p_local) {
  const int d = gd.d;
  double* xL = workV[0];
  const bool fused = fusable();
  if (fused) {
    // small grids (launch bound): the gradient's loader reads the global vector itself, zero Dirichlet rows filled on the fly
    // (:635-637 + :639 in one launch); large grids keep the padded copy, whose 16-byte block loads are cheaper than the gather
    const bool fuse_pad = gd.m <= SB200_FUSE_PAD_MAX_NODES;
    if (!fuse_pad) SB_TRY(pad_vel(x, xstride, xoff, false, xL, s));
    DerivParams jobs[3];
    for (int i = 0; i < d; i++) {
      jobs[i] = job_v(i, fuse_pad ? nullptr : xL, workV[2 + i], nullptr, DERIV_STORE);
      if (fuse_pad) {
        jobs[i].lm = line_map(i, d);
        jobs[i].gsrc = x;
        jobs[i].gs_stride = xstride;
        jobs[i].gs_off = xoff;
      }
    }
    SB_TRY(run_jobs(jobs, d, s));
  } else {
  SB_TRY(pad_vel(x, xstride, xoff, false, xL, s));                                             // :635-637
  if (batchable()) {
    DerivParams jobs[3];
    for (int i = 0; i < d; i++) jobs[i] = job_v(i, xL, workV[2 + i], nullptr, DERIV_STORE);
    SB_TRY(run_jobs(jobs, d, s));
  } else {
    for (int i = 0; i < d; i++) SB_TRY(deriv_v(i, xL, workV[2 + i], nullptr, DERIV_STORE, s));  // :639
  }
  }
  // the divergence rows: inside the flux kernel (from the gradient in its registers) on the fused path, else a pass of their own
  // before the flux overwrites the gradient - the same arithmetic either way
  // the divergence rows: written by the flux kernel from the gradient in its registers (the arithmetic of crop_trace_kernel; decode_node
  // knows the slab view, so this holds on a partition too)
  DivDst dv{nullptr, 0, 0};
  if (div_dst) dv = DivDst{div_dst, div_stride, div_off};
  SB_TRY(join_pressure(s));  // the folded pressure prepared on the side stream
  if (d == 2) {
    VPtrs<2> p;
    for (int j = 0; j < 2; j++) { p.v[j] = workV[2 + j]; p.s[j] = strain[j]; }
    if (p_local) vv_flux_kernel<2, true><<<grid_for(gd.m), 256, 0, s>>>(gd.m, eta, deta, p, p_local, gd, dv);
    else vv_flux_kernel<2><<<grid_for(gd.m), 256, 0, s>>>(gd.m, eta, deta, p, nullptr, gd, dv);
  } else {
    VPtrs<3> p;
    for (int j = 0; j < 3; j++) { p.v[j] = workV[2 + j]; p.s[j] = strain[j]; }
    if (p_local) vv_flux_kernel<3, true><<<grid_for(gd.m), 256, 0, s>>>(gd.m, eta, deta, p, p_local, gd, dv);
    else vv_flux_kernel<3><<<grid_for(gd.m), 256, 0, s>>>(gd.m, eta, deta, p, nullptr, gd, dv);
  }
  count_launch();
  SB_CUDA(cudaGetLastError());
  return viscous_tail(dst, dstride, doff, s);
}

int StokesCtx::divergence_into(const double* x, int xstride, int xoff, bool with_dirichlet, double* dst, int dstride,
                               int doff, cudaStream_t s) {
  const int d = gd.d;
  double* xL = workV[0];
  if (fusable() && gd.m <= SB200_FUSE_CROP_MAX_NODES) {
    // one launch: D_i v_i for i < d-1 stored as terms, the last axis' epilogue applies the "+=" chain (:584-590) and scatters (:592);
    // with zero boundary rows the loaders read the global vector directly, with Dirichlet data the padded copy is made first
    const bool fuse_pad = !with_dirichlet && gd.m <= SB200_FUSE_PAD_MAX_NODES;
    if (!fuse_pad) SB_TRY(pad_vel(x, xstride, xoff, with_dirichlet, xL, s));  // :574-581
    double* terms[2] = {workP[1], workP[2]};  // (workP[0] may hold the folded pressure of the caller)
    DerivParams jobs[3];
    for (int i = 0; i < d; i++) {
      jobs[i] = job_p(i, xL, d, i, i < d - 1 ? terms[i] : nullptr, 1, 0, nullptr, DERIV_STORE);
      if (fuse_pad) {
        jobs[i].lm = line_map(i, 1);
        jobs[i].gsrc = x;
        jobs[i].gs_stride = xstride;
        jobs[i].gs_off = xoff + i;
      }
    }
    DerivParams& f = jobs[d - 1];
    f.lm = line_map(d - 1, 1);
    f.gdst = dst;
    f.gd_stride = dstride;
    f.gd_off = doff;
    f.fin = EO_FIN_SUM;
    f.nterms = d - 1;
    for (int i = 0; i < d - 1; i++) f.term[i] = terms[i];
    f.sign = 1.0;
    return run_jobs(jobs, d, s);
  }
  SB_TRY(pad_vel(x, xstride, xoff, with_dirichlet, xL, s));  // :574-581
  if (fusable() || batchable()) {
    // one launch for the d terms D_i v_i; the "+=" chain (stokes.C:584-590) is applied by the crop in axis order
    double* terms[3] = {workP[0], workP[1], workP[2]};
    DerivParams jobs[3];
    for (int i = 0; i < d; i++) jobs[i] = job_p(i, xL, d, i, terms[i], 1, 0, nullptr, DERIV_STORE);
    SB_TRY(run_jobs(jobs, d, s));
    return crop_sum(1, d, terms, 1.0, dst, dstride, doff, s);
  }
  double* acc = workP[2];
  for (int i = 0; i < d; i++)  // :584-590  component i gathered by stride, accumulated in the epilogue
    SB_TRY(deriv_p(i, xL, d, i, acc, 1, 0, i == 0 ? nullptr : acc, DERIV_ADD, s));
  return crop(1, acc, dst, dstride, doff, false, nullptr, s);  // :592
}

// pL = the padded, boundary-extrapolated pressure of a global vector (stokes.C:606-609): pad + StokesPressureReduceOrder.
int StokesCtx::pad_pres_reduced(const double* src, int sstride, int soff, double* pL, cudaStream_t s) {
  const int d = gd.d;
  if (d >= 2 && gd.stride[d - 1] == 1 && gdim[d - 1] >= 3 && gd.m < (1ll << 31)) {
    const long long nlines = gd.m / gd.dim[d - 1];
    pad_reduce_lastaxis_kernel<<<(unsigned)((nlines * 32 + 255) / 256), 256, 0, s>>>(gd, src, sstride, soff, w0[d - 1], w1[d - 1], pL);
    count_launch();
    SB_CUDA(cudaGetLastError());
    return pressure_reduce_order(pL, s, 1);  // the remaining passes
  }
  SB_TRY(pad_pres(src, sstride, soff, pL, s));
  return pressure_reduce_order(pL, s);
}

// The folded pressure of StokesMatMult / StokesFunction (workP[0]): on one GPU prepared on the side stream while the caller's stream pads
// and differentiates the velocity; the consumer (flux / rheology kernel) joins through join_pressure().  On a slab partition the
// extrapolation contains cross-rank barriers, which must stay in the one stream order every rank shares: serial there.
int StokesCtx::fold_pressure_begin(const double* xG, cudaStream_t s) {
  const int d = gd.d;
  if (arena.nranks == 1) {
    SB_CUDA(cudaEventRecord(ev_fork, s));
    SB_CUDA(cudaStreamWaitEvent(aux_stream, ev_fork, 0));
    SB_TRY(pad_pres_reduced(xG, d + 1, d, workP[0], aux_stream));
    SB_CUDA(cudaEventRecord(ev_pjoin, aux_stream));
    pressure_pending = true;
    return 0;
  }
  return pad_pres_reduced(xG, d + 1, d, workP[0], s);
}

int StokesCtx::join_pressure(cudaStream_t s) {
  if (pressure_pending) {
    SB_CUDA(cudaStreamWaitEvent(s, ev_pjoin, 0));
    pressure_pending = false;
  }
  return 0;
}

int StokesCtx::pressure_reduce_order(double* pL, cudaStream_t s, int first_pass) {
  // stokes.C:1029-1080: z lines, then y lines, then x lines; later passes consume earlier results
  const int d = gd.d;
  const bool slab = arena.nranks > 1;
  for (int pass = first_pass; pass < d; pass++) {
    const int axis = d - 1 - pass;
    if (gdim[axis] < 3) continue;
    if (axis == 0 && slab) {
      // the partitioned axis: partial sums per rank, pushed to the two end-plane owners and added in rank order
      SB_CHECK(arena.attached(), SB200_ERR_USER, "slab partition: peers are not attached (exchange the IPC handles first)");
      const long long R0 = gd.stride[0];
      const int G = arena.nranks, P = gdim[0];
      double* mine_on_first = arena.on(0, red) + (size_t)arena.rank * 2 * R0;
      double* mine_on_last = arena.on(G - 1, red) + (size_t)arena.rank * 2 * R0;
      reduce0_partial_kernel<<<(unsigned)((R0 + 127) / 128), 128, 0, s>>>(w0[0], w1[0], pL, gd.i0, gd.dim[0], P, R0, mine_on_first, mine_on_last);
      count_launch();
      SB_CUDA(cudaGetLastError());
      SB_TRY(arena.barrier(s));
      if (arena.rank == 0) {
        reduce0_finish_kernel<<<(unsigned)((R0 + 127) / 128), 128, 0, s>>>(red, G, 0, R0, pL);
        count_launch();
      }
      if (arena.rank == G - 1) {
        reduce0_finish_kernel<<<(unsigned)((R0 + 127) / 128), 128, 0, s>>>(red, G, 1, R0, pL + (size_t)(gd.dim[0] - 1) * R0);
        count_launch();
      }
      SB_CUDA(cudaGetLastError());
      SB_TRY(arena.barrier(s));  // the slots may be overwritten by the next call only after both sums are done
      continue;
    }
    ReduceArgs a;
    a.axis = axis;
    a.P = gd.dim[axis];
    for (int j = 0; j < 3; j++) { a.lo[j] = 0; a.hi[j] = 0; a.stride[j] = 0; }
    for (int j = 0; j < d; j++) {
      a.stride[j] = gd.stride[j];
      // axes slower than `axis` were not extended yet: interior only; faster ones already were: full range
      int lo = (j < axis) ? 1 : 0;
      int hi = (j < axis) ? gd.gext(j) - 2 : gd.gext(j) - 1;
      if (j == 0) {  // clip the global plane range to this rank's slab (local indices)
        lo = std::max(lo, gd.i0) - gd.i0;
        hi = std::min(hi, gd.i0 + gd.dim[0] - 1) - gd.i0;
      }
      a.lo[j] = lo;
      a.hi[j] = hi;
    }
    a.nother = 0;
    a.nlines = 1;
    bool empty = false;
    for (int j = 0; j < d; j++)
      if (j != axis) {
        a.oax[a.nother++] = j;
        if (a.hi[j] < a.lo[j]) empty = true;
        a.nlines *= (a.hi[j] - a.lo[j] + 1);
      }
    if (empty || a.nlines <= 0) continue;
    if (axis == d - 1 && gd.stride[axis] == 1)
      reduce_order_lastaxis_kernel<<<(unsigned)((a.nlines * 32 + 255) / 256), 256, 0, s>>>(a, w0[axis], w1[axis], pL);
    else
      reduce_order_kernel<<<(unsigned)((a.nlines + 31) / 32), dim3(32, 8), 0, s>>>(a, w0[axis], w1[axis], pL);
    count_launch();
    SB_CUDA(cudaGetLastError());
  }
  return 0;
}

int StokesCtx::matmult_vp_into(const double* x, int xstride, int xoff, double* dst, int dstride, int doff, bool add,
                               const double* sub, cudaStream_t s) {
  const int d = gd.d;
  double* pL = workP[0];
  SB_TRY(pad_pres_reduced(x, xstride, xoff, pL, s));  // :606-609
  double* vL = workV[0];
  if (fusable()) {
    // D_i p goes straight into component i of the global velocity rows (:611-617), with the caller's "+=" / "- force" applied there
    DerivParams jobs[3];
    for (int i = 0; i < d; i++) {
      jobs[i] = job_p(i, pL, 1, 0, nullptr, 1, 0, nullptr, DERIV_STORE);
      jobs[i].lm = line_map(i, 1);
      jobs[i].gdst = dst;
      jobs[i].gd_stride = dstride;
      jobs[i].gd_off = doff + i;
      jobs[i].fin = EO_FIN_RAW;
      jobs[i].add = add ? 1 : 0;
      jobs[i].sub = sub;
    }
    return run_jobs(jobs, d, s);
  }
  if (batchable()) {
    DerivParams jobs[3];
    for (int i = 0; i < d; i++) jobs[i] = job_p(i, pL, 1, 0, vL, d, i, nullptr, DERIV_STORE);
    SB_TRY(run_jobs(jobs, d, s));
  } else {
    for (int i = 0; i < d; i++) SB_TRY(deriv_p(i, pL, 1, 0, vL, d, i, nullptr, DERIV_STORE, s));  // :611-614
  }
  return crop(d, vL, dst, dstride, doff, add, sub, s);                                         // :617
}

int StokesCtx::matmult(const double* xG, double* yG, cudaStream_t s) {
  SB_CHECK(xG && yG && xG != yG, SB200_ERR_ARG, "StokesMatMult: x and y must be distinct non-null vectors");
  const int d = gd.d;
  const double* pfold = nullptr;
  if (fold_pressure) {  // opt-in: the padded, boundary-extrapolated pressure (:606-609) enters the viscous flux as -p I
    SB_TRY(fold_pressure_begin(xG, s));
    pfold = workP[0];
  }
  if (trace_divergence) {
    SB_TRY(matmult_vv_into(xG, d + 1, 0, yG, d + 1, 0, s, yG, d + 1, d, pfold));  // :508-509  vG1 = VV v and pG1 = PV v from one gradient
  } else {
    SB_TRY(matmult_vv_into(xG, d + 1, 0, yG, d + 1, 0, s, nullptr, 0, 0, pfold));  // :508  vG1 = VV v
    SB_TRY(divergence_into(xG, d + 1, 0, false, yG, d + 1, d, s));                 // :509  pG1 = PV v (workP is free again by now)
  }
  if (!fold_pressure) SB_TRY(matmult_vp_into(xG, d + 1, d, yG, d + 1, 0, true, nullptr, s));  // :512-513  vG1 += VP p
  return 0;
}

int StokesCtx::function(const double* xG, double* yG, cudaStream_t s) {
  SB_CHECK(xG && yG && xG != yG, SB200_ERR_ARG, "StokesFunction: x and y must be distinct non-null vectors");
  const int d = gd.d;
  double* xL = workV[0];
  const double* pfold = nullptr;
  if (fold_pressure) {  // as in matmult(): V = eta*eps - p I, so the viscous tail also yields the pressure gradient (:747-750); prepared
    SB_TRY(fold_pressure_begin(xG, s));  // first (on one GPU on the side stream, beside the velocity pad and the gradient batch)
    pfold = workP[0];
  }
  SB_TRY(pad_vel(xG, d + 1, 0, true, xL, s));                                                 // :691-699
  if (fusable() || batchable()) {
    DerivParams jobs[3];
    for (int i = 0; i < d; i++) jobs[i] = job_v(i, xL, strain[i], nullptr, DERIV_STORE);
    SB_TRY(run_jobs(jobs, d, s));
  } else {
    for (int i = 0; i < d; i++) SB_TRY(deriv_v(i, xL, strain[i], nullptr, DERIV_STORE, s));   // :701
  }
  DivDst dv{nullptr, 0, 0};  // :746 from the gradient above (same Dirichlet-padded input): inside the rheology kernel on the fused path
  if (trace_divergence) dv = DivDst{yG, d + 1, d};
  SB_TRY(join_pressure(s));
  init_minmax_kernel<<<1, 1, 0, s>>>(minmax);
  count_launch();
  Rheo r{rheology, hardness, exponent, regularization, gamma0};
  if (d == 2) {
    VPtrs<2> p;
    for (int j = 0; j < 2; j++) { p.v[j] = workV[2 + j]; p.s[j] = strain[j]; }
    if (pfold) rheology_kernel<2, true><<<grid_for(gd.m), 256, 0, s>>>(gd.m, r, eta, deta, p, minmax, pfold, gd, dv);
    else rheology_kernel<2><<<grid_for(gd.m), 256, 0, s>>>(gd.m, r, eta, deta, p, minmax, nullptr, gd, dv);
  } else {
    VPtrs<3> p;
    for (int j = 0; j < 3; j++) { p.v[j] = workV[2 + j]; p.s[j] = strain[j]; }
    if (pfold) rheology_kernel<3, true><<<grid_for(gd.m), 256, 0, s>>>(gd.m, r, eta, deta, p, minmax, pfold, gd, dv);
    else rheology_kernel<3><<<grid_for(gd.m), 256, 0, s>>>(gd.m, r, eta, deta, p, minmax, nullptr, gd, dv);
  }
  count_launch();
  SB_CUDA(cudaGetLastError());
  SB_TRY(viscous_tail(yG, d + 1, 0, s));                                // :737-744 -> velocity slots
  if (!trace_divergence) SB_TRY(divergence_into(xG, d + 1, 0, true, yG, d + 1, d, s));  // :746 -> pressure slots
  if (!fold_pressure) SB_TRY(matmult_vp_into(xG, d + 1, d, yG, d + 1, 0, true, nullptr, s));  // :747-750
  // :756 yG -= force
  {
    SB_TRY(axpy_launch(g, -1.0, force, yG, s));
  }
  return 0;
}

int StokesCtx::get_diagonal_schur(double* y, cudaStream_t s) {
  recip_crop_kernel<<<grid_for(gd.m), 256, 0, s>>>(gd, eta, y);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return 0;
}

int StokesCtx::matmult_schur(const double* x, double* y, sb200_velocity_solve_fn solve, void* solve_ctx, cudaStream_t s) {
  SB_CHECK(solve, SB200_ERR_ARG, "StokesMatMultSchur needs the inner velocity solve (KSPSchurVelocity, stokes.C:531)");
  SB_TRY(matmult_vp_into(x, 1, 0, vG0, gd.d, 0, false, nullptr, s));  // :530
  int rc = solve(solve_ctx, vG0, vG1, (void*)s);                      // :531
  SB_CHECK(rc == 0, rc, "inner velocity solve failed");
  SB_TRY(divergence_into(vG1, gd.d, 0, false, y, 1, 0, s));  // :532
  scale_kernel<<<grid_for(gp), 256, 0, s>>>(gp, -1.0, y);     // :533
  count_launch();
  SB_CUDA(cudaGetLastError());
  return 0;
}

namespace {
__global__ void axpy_kernel(long long n, double a, const double* __restrict__ x, double* __restrict__ y) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) y[i] = y[i] + a * x[i];
}
}  // namespace

int axpy_launch(long long n, double a, const double* x, double* y, cudaStream_t s) {
  axpy_kernel<<<grid_for(n), 256, 0, s>>>(n, a, x, y);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace sb200
