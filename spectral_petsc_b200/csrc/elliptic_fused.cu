// Fused MatMult_Elliptic (elliptic.C:297-339) for d-dimensional grids whose extents are all P with
// P % 16 == 0 (P = 32, 64, 128): one persistent "chain" kernel per axis,
//     out  = 0   - D_0 (eta D_0 w + deta w g0_0)          axis 0   (FIRST: no read of out)
//     out  = out - D_k (eta D_k w + deta w g0_k)          middle axes
//     V    = crop(out - D_l (eta D_l w + deta w g0_l))    last axis (R == 1; crop fused)
// preserving the reference's accumulation order (elliptic.C:331-334).  Each warp runs the whole
// chain for 8 grid lines out of shared memory (see chain.cuh); the even-odd halves of D are resident
// in shared memory for the life of the persistent CTA.
#include "../../include/spectral_b200.h"
#include "chain.cuh"
#include "deriv.h"
#include "elliptic.h"

namespace sb200 {

namespace {

constexpr int NWARPS = 16;

struct ChainParams {
  const double* Ae;
  const double* Bo;
  const double* w;     // padded local field (m)
  const double* eta;   // m
  const double* deta;  // m
  const double* g0;    // gradu[axis] (m)
  double* out;         // m: accumulator field
  double* V;           // g: cropped result (LAST only)
  LineGeom lg;
  // crop geometry (LAST): lines are indexed by the leading d-1 indices
  int d;
  int dim[SB200_MAX_DIM];
};

enum { POS_FIRST = 0, POS_MID = 1, POS_LAST = 2 };

template <int P, bool RIGHT, int POS>
__global__ void __launch_bounds__(NWARPS * 32, 1) chain_kernel(ChainParams p) {
  using E = EO<P>;
  extern __shared__ double sm[];
  double* Ae = sm;
  double* Bo = sm + E::H * E::LDM;
  constexpr int BE = RIGHT ? E::BLOCK_ELEMS_RIGHT : E::BLOCK_ELEMS_LEFT;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  double* Xw = sm + E::MAT_ELEMS + warp * BE;

  const long long nblocks = p.lg.nlines / 8;  // host guarantees nlines % 8 == 0
  const long long per = (nblocks + gridDim.x - 1) / gridDim.x;
  const long long b_begin = (long long)blockIdx.x * per;
  const long long b_end = b_begin + per < nblocks ? b_begin + per : nblocks;

  load_matrices<P>(sm, p.Ae, p.Bo);
  long long blk = b_begin + warp;
  if (blk < b_end) load_block<P, RIGHT>(Xw, p.w, p.lg, blk * 8, lane);
  cp_async_wait<0>();
  __syncthreads();  // matrices visible to all warps (the only CTA-wide barrier)

  for (; blk < b_end; blk += NWARPS) {
    const long long n0 = blk * 8;
    const long long base0 = RIGHT ? n0 * P : p.lg.base(n0);
    Own<P, RIGHT> own;
    own.base = RIGHT ? (n0 + g) * P : base0 + 2 * t;
    own.R = p.lg.R;
    own.g = g;
    own.t = t;
    // pull the epilogue operands of this block towards L2 while the tensor pipe works
    prefetch_block<P, RIGHT>(p.eta, base0, p.lg.R, lane);
    prefetch_block<P, RIGHT>(p.deta, base0, p.lg.R, lane);
    prefetch_block<P, RIGHT>(p.g0, base0, p.lg.R, lane);
    if (POS != POS_FIRST) prefetch_block<P, RIGHT>(p.out, base0, p.lg.R, lane);

    double a[E::MT][2], b[E::MT][2];
    eo_gemm<P, RIGHT>(Ae, Bo, Xw, a, b, g, t);
    __syncwarp();
    // flux (elliptic.C:319-323) written back in place: f = eta*y + (deta*w)*g0 ; loads batched 2 tiles deep
#pragma unroll
    for (int ib = 0; ib < E::MT; ib += 2) {
      double2 e[2][2], de[2][2], gg[2][2];
#pragma unroll
      for (int ii = 0; ii < 2; ii++) {
        const long long ot = own.top(ib + ii), ob = own.bot(ib + ii);
        e[ii][0] = ldg2(p.eta + ot);
        e[ii][1] = ldg2(p.eta + ob);
        de[ii][0] = ldg2(p.deta + ot);
        de[ii][1] = ldg2(p.deta + ob);
        gg[ii][0] = ldg2(p.g0 + ot);
        gg[ii][1] = ldg2(p.g0 + ob);
      }
#pragma unroll
      for (int ii = 0; ii < 2; ii++) {
        const int i = ib + ii;
        const int st = own.stop(i), sb = own.sbot(i);
        const double2 wt = ld2(Xw + st), wb = ld2(Xw + sb);
        const double yt0 = a[i][0] + b[i][0], yt1 = a[i][1] + b[i][1];
        const double yb0 = RIGHT ? b[i][1] - a[i][1] : b[i][0] - a[i][0];
        const double yb1 = RIGHT ? b[i][0] - a[i][0] : b[i][1] - a[i][1];
        const double ft0 = __dadd_rn(__dmul_rn(e[ii][0].x, yt0), __dmul_rn(__dmul_rn(de[ii][0].x, wt.x), gg[ii][0].x));
        const double ft1 = __dadd_rn(__dmul_rn(e[ii][0].y, yt1), __dmul_rn(__dmul_rn(de[ii][0].y, wt.y), gg[ii][0].y));
        const double fb0 = __dadd_rn(__dmul_rn(e[ii][1].x, yb0), __dmul_rn(__dmul_rn(de[ii][1].x, wb.x), gg[ii][1].x));
        const double fb1 = __dadd_rn(__dmul_rn(e[ii][1].y, yb1), __dmul_rn(__dmul_rn(de[ii][1].y, wb.y), gg[ii][1].y));
        st2(Xw + st, ft0, ft1);
        st2(Xw + sb, fb0, fb1);
      }
    }
    __syncwarp();
    eo_gemm<P, RIGHT>(Ae, Bo, Xw, a, b, g, t);
    __syncwarp();  // all lanes done reading the block: safe to refill it
    const long long nblk = blk + NWARPS;
    if (nblk < b_end) load_block<P, RIGHT>(Xw, p.w, p.lg, nblk * 8, lane);  // overlaps the epilogue

    // epilogue: out = (FIRST ? 0 : out) - D f ; LAST crops into V (LAST is always the R == 1 axis)
    long long vrow = 0;
    bool vint = false;
    if (POS == POS_LAST) {
      // line index = lexicographic index over the leading d-1 axes; interior id of the line
      long long n = n0 + g, gid = 0, mul = 1;
      vint = true;
      for (int j = p.d - 2; j >= 0; j--) {
        const int ij = (int)(n % p.dim[j]);
        n /= p.dim[j];
        vint = vint && ij > 0 && ij < p.dim[j] - 1;
        gid += (long long)(ij - 1) * mul;
        mul *= p.dim[j] - 2;
      }
      vrow = gid * (P - 2) - 1;  // V index of row m is vrow + m
    }
#pragma unroll
    for (int ib = 0; ib < E::MT; ib += 4) {
      double2 ot[4], ob[4];
      if (POS != POS_FIRST) {
#pragma unroll
        for (int ii = 0; ii < 4; ii++) {
          if (ib + ii >= E::MT) continue;  // (MT % 4 != 0: the last batch is short)
          ot[ii] = ld2(p.out + own.top(ib + ii));
          ob[ii] = ld2(p.out + own.bot(ib + ii));
        }
      } else {
#pragma unroll
        for (int ii = 0; ii < 4; ii++) ot[ii] = ob[ii] = make_double2(0.0, 0.0);
      }
#pragma unroll
      for (int ii = 0; ii < 4; ii++) {
        const int i = ib + ii;
        if (i >= E::MT) continue;
        const double yt0 = a[i][0] + b[i][0], yt1 = a[i][1] + b[i][1];
        const double yb0 = RIGHT ? b[i][1] - a[i][1] : b[i][0] - a[i][0];
        const double yb1 = RIGHT ? b[i][0] - a[i][0] : b[i][1] - a[i][1];
        const double rt0 = ot[ii].x - yt0, rt1 = ot[ii].y - yt1;
        const double rb0 = ob[ii].x - yb0, rb1 = ob[ii].y - yb1;
        if (POS != POS_LAST) {
          st2(p.out + own.top(i), rt0, rt1);
          st2(p.out + own.bot(i), rb0, rb1);
        } else if (vint) {
          const int mt = i * 8 + 2 * t, mb = P - 2 - i * 8 - 2 * t;  // first row of each pair
          if (mt > 0) p.V[vrow + mt] = rt0;
          p.V[vrow + mt + 1] = rt1;  // mt+1 <= P/2 - 1
          p.V[vrow + mb] = rb0;      // mb >= P/2
          if (mb + 1 < P - 1) p.V[vrow + mb + 1] = rb1;
        }
      }
    }
    if (nblk < b_end) cp_async_wait<0>();
    __syncwarp();
  }
}

template <int P, bool RIGHT, int POS>
int launch_chain(const ChainParams& p, cudaStream_t s) {
  using E = EO<P>;
  constexpr int BE = RIGHT ? E::BLOCK_ELEMS_RIGHT : E::BLOCK_ELEMS_LEFT;
  const size_t smem = (size_t)(E::MAT_ELEMS + NWARPS * BE) * sizeof(double);
  auto kern = chain_kernel<P, RIGHT, POS>;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  static bool attr[64] = {};  // the opt-in above 48 KB of dynamic shared memory is per device
  if (!attr[dev & 63]) {
    SB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr[dev & 63] = true;
  }
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const long long nblocks = p.lg.nlines / 8;
  // one persistent CTA per SM; fewer when there is not a block per warp to hand out
  long long grid = (nblocks + NWARPS - 1) / NWARPS;
  if (grid > sms) grid = sms;
  if (grid < 1) grid = 1;
  kern<<<(unsigned)grid, NWARPS * 32, smem, s>>>(p);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return 0;
}

template <int P>
int matmult_fused_P(EllipticCtx& e, const double* U, double* V, cudaStream_t s) {
  const int d = e.gd.d;
  SB_TRY(e.pad(U, false, e.w[0], s));
  for (int k = 0; k < d; k++) {
    ChainParams p;
    p.Ae = e.Dax[k]->d_Ae;
    p.Bo = e.Dax[k]->d_Bo;
    p.w = e.w[0];
    p.eta = e.eta;
    p.deta = e.deta;
    p.g0 = e.gradu[k];
    p.out = e.w[1];
    p.V = V;
    p.lg.R = e.gd.stride[k];
    p.lg.PR = (long long)P * e.gd.stride[k];
    p.lg.nlines = e.gd.m / P;
    p.d = d;
    for (int j = 0; j < d; j++) p.dim[j] = e.gd.dim[j];
    const bool last = (k == d - 1);
    if (k == 0 && !last) SB_TRY((launch_chain<P, false, POS_FIRST>(p, s)));
    else if (!last) SB_TRY((launch_chain<P, false, POS_MID>(p, s)));
    else SB_TRY((launch_chain<P, true, POS_LAST>(p, s)));
  }
  return 0;
}

}  // namespace

bool elliptic_fused_supported(const EllipticCtx& e) {
  const int d = e.gd.d;
  if (d < 2) return false;
  const int P = e.gd.dim[0];
  for (int j = 1; j < d; j++)
    if (e.gd.dim[j] != P) return false;
  return (P == 32 || P == 64 || P == 128) && (e.gd.m / P) % 8 == 0;
}

int elliptic_matmult_fused(EllipticCtx& e, const double* U, double* V, cudaStream_t s) {
  switch (e.gd.dim[0]) {
    case 32: return matmult_fused_P<32>(e, U, V, s);
    case 64: return matmult_fused_P<64>(e, U, V, s);
    case 128: return matmult_fused_P<128>(e, U, V, s);
  }
  set_last_error("fused path: unsupported extent");
  return SB200_ERR_SUP;
}

}  // namespace sb200
