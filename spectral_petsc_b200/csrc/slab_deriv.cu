// Derivative along the partitioned axis 0 of a slab-distributed field, transpose based:
//   push   : every rank stores its planes of the operand into the column pencils of all ranks  (all-to-all #1)
//   local  : each rank differentiates its pencil (all P planes of R/G columns) with the ordinary kernels
//   push   : every rank stores its result rows into the slabs of the planes' owners             (all-to-all #2)
// with one device-side barrier after each push.  Per rank 2 * 8 B * (G-1)/G of the field cross NVLink, against
// (G-1)/G of the WHOLE field per rank for the operand-pull scheme (deriv_generic.cu slab mode), which this replaces
// whenever the column count divides by the number of ranks.  The "field" is the scalar view (P planes x R columns,
// element stride / offset for AoS components) that DerivParams describes.
#include "../../include/spectral_b200.h"
#include "common.cuh"
#include "deriv.h"
#include "symm.h"

namespace sb200 {

namespace {

struct PushPtrs {
  double* dst[SB200_MAX_RANKS];
};

// Xp_q[(i0 + ml) * Rp + (c - q*Rp)] = x[(ml*R + c) * xs + xoff]        ml < nloc, c < R
__global__ void __launch_bounds__(256) push_to_pencils_kernel(const double* __restrict__ x, int xs, int xoff, PushPtrs pp, int nloc, int i0,
                                                              long long R, long long Rp) {
  const long long total = (long long)nloc * R, stride = (long long)gridDim.x * blockDim.x;
  for (long long e0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; e0 < total; e0 += 4 * stride) {
    double v[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const long long e = e0 + u * stride;
      v[u] = e < total ? x[e * xs + xoff] : 0.0;
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const long long e = e0 + u * stride;
      if (e >= total) continue;
      const long long ml = e / R, c = e - ml * R;
      const int q = (int)(c / Rp);
      pp.dst[q][(i0 + ml) * Rp + (c - q * Rp)] = v[u];
    }
  }
}

// y_q[((k - q*nloc) * R + rank*Rp + c) * ys + yoff] (op)= Yp[k * Rp + c]      k < P, c < Rp, q = k / nloc
__global__ void __launch_bounds__(256) push_to_slabs_kernel(const double* __restrict__ Yp, PushPtrs pp, int ys, int yoff, int P, int nloc,
                                                            int rank, long long R, long long Rp, int negate) {
  const long long total = (long long)P * Rp, stride = (long long)gridDim.x * blockDim.x;
  for (long long e0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; e0 < total; e0 += 4 * stride) {
    double v[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const long long e = e0 + u * stride;
      v[u] = e < total ? Yp[e] : 0.0;
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const long long e = e0 + u * stride;
      if (e >= total) continue;
      const long long k = e / Rp, c = e - k * Rp;
      const int q = (int)(k / nloc);
      pp.dst[q][((k - (long long)q * nloc) * R + (long long)rank * Rp + c) * ys + yoff] = negate ? 0.0 - v[u] : v[u];
    }
  }
}

int blocks_for(long long n) {
  long long b = (n + 1023) / 1024;
  if (b > 148 * 8) b = 148 * 8;
  return (int)(b < 1 ? 1 : b);
}

}  // namespace

bool slab_deriv0_pencil_supported(const SymmArena& a, const DerivParams& p) {
  // accumulation onto an existing field would need the old values at the destination: only "y = D x",
  // "y = 0 - D x" and "y = 0 + D x" (the first step of the reference's AXPY chains) are handled here
  return a.nranks > 1 && p.O == 1 && p.R % a.nranks == 0 && (p.mode == DERIV_STORE || p.yin == nullptr);
}

// p: the slab-local description (x, y local arena arrays of this rank; O == 1; P = global extent; R columns).
// Xp, Yp: arena arrays of at least P * R / nranks doubles.
int slab_deriv0_pencil(SymmArena& a, const DerivParams& p, int nloc, int i0, double* Xp, double* Yp, cudaStream_t s) {
  SB_CHECK(a.attached(), SB200_ERR_USER, "slab partition: peers are not attached (exchange the IPC handles first)");
  const int G = a.nranks;
  const long long R = p.R, Rp = R / G;
  PushPtrs px;
  for (int q = 0; q < SB200_MAX_RANKS; q++) px.dst[q] = q < G ? a.on(q, Xp) : nullptr;
  push_to_pencils_kernel<<<blocks_for((long long)nloc * R), 256, 0, s>>>(p.x, p.xs, p.xoff, px, nloc, i0, R, Rp);
  count_launch();
  SB_CUDA(cudaGetLastError());
  PushPtrs py;
  for (int q = 0; q < SB200_MAX_RANKS; q++) py.dst[q] = q < G ? a.on(q, p.y) : nullptr;
  SB_TRY(a.barrier(s));
  DerivParams lp = p;  // the pencil: all P planes of Rp columns, unit stride
  lp.x = Xp;
  lp.y = Yp;
  lp.yin = nullptr;
  lp.mode = DERIV_STORE;
  lp.R = Rp;
  lp.xs = lp.ys = 1;
  lp.xoff = lp.yoff = 0;
  lp.npeer = 0;
  // unit-stride result in an aligned even column range: the derivative's epilogue stores the rows straight into the plane owners'
  // fields over NVLink (no pencil result buffer, no second push kernel); otherwise the pencil result goes through push_to_slabs_kernel
  if (p.ys == 1 && p.yoff == 0 && p.sync && Rp % 8 == 0 && R % 2 == 0 && deriv_eo_supported(lp) &&
      reinterpret_cast<uintptr_t>(Xp) % 16 == 0 && reinterpret_cast<uintptr_t>(p.y) % 16 == 0) {
    lp.y = nullptr;
    lp.peer_on = 1;
    lp.peer_nloc = nloc;
    lp.peer_negate = p.mode == DERIV_SUB ? 1 : 0;
    lp.peer_R = R;
    lp.peer_col0 = (long long)a.rank * Rp;
    for (int q = 0; q < G; q++) lp.ypeer[q] = py.dst[q];
    SB_TRY(deriv_eo_apply(lp, p.sync, s));
    return a.barrier(s);
  }
  SB_TRY(deriv_apply(lp, s));
  push_to_slabs_kernel<<<blocks_for((long long)p.P * Rp), 256, 0, s>>>(Yp, py, p.ys, p.yoff, p.P, nloc, a.rank, R, Rp, p.mode == DERIV_SUB ? 1 : 0);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return a.barrier(s);
}

}  // namespace sb200
