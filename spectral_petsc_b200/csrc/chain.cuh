// Warp-private even-odd DMMA machinery for the fused "chain" kernels.
//
// A chain along one axis is  out (-)= D * flux(D * w)  for every grid line of that axis
// (MatMult_Elliptic's  w[1+d] = D_d w0 ; pointwise ; w0 -= D_d w[1+d],  elliptic.C:309-334).
// One warp owns a block of 8 lines (all P points of each) in shared memory and runs the whole
// chain on it with no CTA-level synchronisation:
//     GEMM1 (DMMA)  ->  flux in registers  ->  overwrite the block in place  ->  GEMM2 (DMMA)  ->  epilogue.
//
// Even-odd split: the CGL matrix is centro-antisymmetric, D[n-i][n-j] = -D[i][j] (n = P-1), so with
//   s_j = u_j + u_{n-j},  d_j = u_j - u_{n-j},  Ae = (D[i][j] + D[i][n-j])/2,  Bo = (D[i][j] - D[i][n-j])/2
//   a = Ae s,  b = Bo d   (two h x h products, h = P/2)      y_i = a_i + b_i,   y_{n-i} = b_i - a_i
// which halves the executed flops of the dense P x P product.  s and d are formed on the fly from the
// two shared-memory loads that feed the B fragments; Ae/Bo stay resident in shared memory.
#pragma once
#include "common.cuh"
#include "persist.h"

namespace sb200 {

template <int P>
struct EO {
  static constexpr int H = P / 2;        // pair count
  static constexpr int MT = H / 8;       // m-tiles of pair rows
  static constexpr int KS = H / 4;       // k4 steps
  static constexpr int LDM = H + 4;      // matrix leading dim in smem: (4g+t) mod 16 distinct
  static constexpr int LDR = P + 4;      // RIGHT block leading dim
  static constexpr int MAT_ELEMS = 2 * H * LDM;
  static constexpr int BLOCK_ELEMS_LEFT = P * 8;
  static constexpr int BLOCK_ELEMS_RIGHT = 8 * LDR;
  static_assert(P % 16 == 0, "even-odd DMMA path needs P % 16 == 0");
};

// Shared-memory address of element (row m along the axis, line c in 0..7) of a warp's block.
template <int P, bool RIGHT>
__device__ __forceinline__ int xaddr(int m, int c) {
  if (RIGHT) return c * EO<P>::LDR + m;
  return m * 8 + (c ^ (((m >> 1) & 1) << 2));  // XOR swizzle keeps the B-fragment loads conflict free
}

// a[i], b[i] = Ae * s, Bo * d  for the warp's 8 lines (i = tile of 8 pair indices).
// LEFT  (!RIGHT): matrices are the A operand.  acc[i][h] <-> pair index i*8+g, line 2t+h.
// RIGHT:          the field is the A operand.   acc[i][h] <-> line g, pair index i*8+2t+h.
// Either way a thread's two values are adjacent in global memory (16-byte accesses).
// (Defined after eo_gemm_nt, which it wraps, so that every fused path shares one summation order.)
template <int P, bool RIGHT>
__device__ __forceinline__ void eo_gemm(const double* __restrict__ Ae, const double* __restrict__ Bo,
                                        const double* __restrict__ Xw, double (&a)[EO<P>::MT][2],
                                        double (&b)[EO<P>::MT][2], int g, int t);

// NT-block variant: one set of matrix fragments feeds NT line-blocks (block j at Xw + j*BE).
// Tile range: only the TN pair tiles [i0, i0 + TN) are accumulated (acc[j][i] <-> tile i0 + i), so that two warps can split one
// item's M dimension; every element keeps the k-loop of the whole-item product.
// SB200_KSPLIT == 2: even and odd k-steps accumulate into two independent register sets that are added at the end - 2 x 2 x MT x NT
// independent DMMAs between dependent ones, enough for ONE warp to keep the FP64 tensor pipe busy (the dependent-issue latency of a
// DMMA is ~370 clk = 23 issue slots, profiles/r02_notes.md); costs 4*MT*NT more registers and changes the summation order.
#ifndef SB200_KSPLIT
#define SB200_KSPLIT 1
#endif
template <int P, int NT, bool RIGHT, int TN = EO<P>::MT>
__device__ __forceinline__ void eo_gemm_nt(const double* __restrict__ Ae, const double* __restrict__ Bo,
                                           const double* __restrict__ Xw, double (&a)[NT][TN][2],
                                           double (&b)[NT][TN][2], int g, int t, int i0 = 0) {
  using E = EO<P>;
  constexpr int BE = RIGHT ? E::BLOCK_ELEMS_RIGHT : E::BLOCK_ELEMS_LEFT;
  constexpr int KSP = (SB200_KSPLIT == 2 && E::KS % 2 == 0) ? 2 : 1;
  Ae += i0 * 8 * E::LDM;
  Bo += i0 * 8 * E::LDM;
  double a1[KSP == 2 ? NT : 1][TN][2], b1[KSP == 2 ? NT : 1][TN][2];
#pragma unroll
  for (int j = 0; j < NT; j++)
#pragma unroll
    for (int i = 0; i < TN; i++) {
      a[j][i][0] = a[j][i][1] = b[j][i][0] = b[j][i][1] = 0.0;
      if (KSP == 2) a1[j][i][0] = a1[j][i][1] = b1[j][i][0] = b1[j][i][1] = 0.0;
    }
#pragma unroll 2
  for (int ks = 0; ks < E::KS; ks++) {
    const int kk = ks * 4 + t;
    double s[NT], d[NT];
#pragma unroll
    for (int j = 0; j < NT; j++) {
      const double p = Xw[j * BE + xaddr<P, RIGHT>(kk, g)];
      const double q = Xw[j * BE + xaddr<P, RIGHT>(P - 1 - kk, g)];
      s[j] = p + q;
      d[j] = p - q;
    }
    double fa[TN], fb[TN];
#pragma unroll
    for (int i = 0; i < TN; i++) {
      fa[i] = Ae[(i * 8 + g) * E::LDM + kk];
      fb[i] = Bo[(i * 8 + g) * E::LDM + kk];
    }
    const bool odd = KSP == 2 && (ks & 1);
#pragma unroll
    for (int i = 0; i < TN; i++) {
#pragma unroll
      for (int j = 0; j < NT; j++) {
        double& a0r = odd ? a1[KSP == 2 ? j : 0][i][0] : a[j][i][0];
        double& a1r = odd ? a1[KSP == 2 ? j : 0][i][1] : a[j][i][1];
        double& b0r = odd ? b1[KSP == 2 ? j : 0][i][0] : b[j][i][0];
        double& b1r = odd ? b1[KSP == 2 ? j : 0][i][1] : b[j][i][1];
        if (RIGHT) {
          dmma884(a0r, a1r, s[j], fa[i]);
          dmma884(b0r, b1r, d[j], fb[i]);
        } else {
          dmma884(a0r, a1r, fa[i], s[j]);
          dmma884(b0r, b1r, fb[i], d[j]);
        }
      }
    }
  }
  if (KSP == 2) {
#pragma unroll
    for (int j = 0; j < NT; j++)
#pragma unroll
      for (int i = 0; i < TN; i++) {
        a[j][i][0] += a1[j][i][0];
        a[j][i][1] += a1[j][i][1];
        b[j][i][0] += b1[j][i][0];
        b[j][i][1] += b1[j][i][1];
      }
  }
}

template <int P, bool RIGHT>
__device__ __forceinline__ void eo_gemm(const double* __restrict__ Ae, const double* __restrict__ Bo,
                                        const double* __restrict__ Xw, double (&a)[EO<P>::MT][2],
                                        double (&b)[EO<P>::MT][2], int g, int t) {
  eo_gemm_nt<P, 1, RIGHT>(Ae, Bo, Xw, reinterpret_cast<double (&)[1][EO<P>::MT][2]>(a), reinterpret_cast<double (&)[1][EO<P>::MT][2]>(b), g, t);
}

// Thread-owned element geometry shared by every epilogue.  For tile i the thread owns a "top" pair
// of adjacent elements and the mirrored "bottom" pair (also adjacent, in reversed order):
//   LEFT : rows mt = i*8+g / mb = P-1-mt, lines 2t,2t+1        -> global offset base0 + m*R + 2t
//   RIGHT: line g, rows i*8+2t,+1 / mirrors P-2-i*8-2t,+1      -> global offset (n0+g)*P + row
// top[h]  <-> acc (a+b)[i][h];   LEFT: bot[h] <-> (b-a)[i][h];   RIGHT: bot[h] <-> (b-a)[i][1-h].
// i counts the warp's own tiles, which start at pair row r0 (0 unless two warps split the item).
template <int P, bool RIGHT>
struct Own {
  long long base;  // LEFT: base0 + 2t ; RIGHT: (n0+g)*P
  long long R;
  int g, t;
  int r0 = 0;
  __device__ __forceinline__ long long top(int i) const {
    return RIGHT ? base + r0 + i * 8 + 2 * t : base + (long long)(r0 + i * 8 + g) * R;
  }
  __device__ __forceinline__ long long bot(int i) const {
    return RIGHT ? base + (P - 2 - r0 - i * 8 - 2 * t) : base + (long long)(P - 1 - r0 - i * 8 - g) * R;
  }
  // shared-memory addresses of the same pairs inside the warp's block (both 16-byte aligned)
  __device__ __forceinline__ int stop(int i) const {
    return RIGHT ? xaddr<P, true>(r0 + i * 8 + 2 * t, g) : xaddr<P, false>(r0 + i * 8 + g, 2 * t);
  }
  __device__ __forceinline__ int sbot(int i) const {
    return RIGHT ? xaddr<P, true>(P - 2 - r0 - i * 8 - 2 * t, g) : xaddr<P, false>(P - 1 - r0 - i * 8 - g, 2 * t);
  }
};

__device__ __forceinline__ double2 ldg2(const double* p) { return __ldg(reinterpret_cast<const double2*>(p)); }
__device__ __forceinline__ double2 ld2(const double* p) { return *reinterpret_cast<const double2*>(p); }
__device__ __forceinline__ void st2(double* p, double x, double y) { *reinterpret_cast<double2*>(p) = make_double2(x, y); }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// Warp-level L2 prefetch of the block's footprint in array x (issued long before the epilogue reads it).
// NPART warps that share the block each prefetch every NPART-th chunk, starting at chunk `part`.
template <int P, bool RIGHT, int NPART = 1>
__device__ __forceinline__ void prefetch_block(const double* __restrict__ x, long long base0, long long R, int lane, int part = 0) {
  if (RIGHT) {
    // 8 lines x P contiguous doubles starting at base0 = n0*P : 8*P*8 bytes = P/2 lines of 128 B
#pragma unroll
    for (int l = lane + 32 * part; l < P / 2; l += 32 * NPART) prefetch_l2(x + base0 + l * 16);
  } else {
#pragma unroll
    for (int m = lane + 32 * part; m < P; m += 32 * NPART) prefetch_l2(x + base0 + (long long)m * R);
  }
}

// Cooperative (whole CTA) load of Ae, Bo ([H][H] row-major in global) into padded smem.
template <int P>
__device__ __forceinline__ void load_matrices(double* sm, const double* __restrict__ gAe, const double* __restrict__ gBo) {
  using E = EO<P>;
  for (int idx = threadIdx.x; idx < E::H * E::H / 2; idx += blockDim.x) {
    const int r = idx / (E::H / 2), c2 = (idx % (E::H / 2)) * 2;
    cp_async16(sm + r * E::LDM + c2, gAe + r * E::H + c2, true);
    cp_async16(sm + E::H * E::LDM + r * E::LDM + c2, gBo + r * E::H + c2, true);
  }
  cp_async_commit();
}

// Line addressing for an array factored as (O, P, R): line n = o*R + r starts at o*P*R + r, stride R.
struct LineGeom {
  long long R, PR, nlines;
  __device__ __forceinline__ long long base(long long n) const {
    const long long o = n / R, r = n - o * R;
    return o * PR + r;
  }
};

// Warp-level load of one 8-line block of field x into Xw (zero fill beyond nlines).
template <int P, bool RIGHT>
__device__ __forceinline__ void load_block(double* Xw, const double* __restrict__ x, const LineGeom& lg,
                                           long long n0, int lane) {
  using E = EO<P>;
  if (RIGHT) {
    // R == 1: each line is P contiguous doubles
#pragma unroll 4
    for (int idx = lane; idx < 8 * (P / 2); idx += 32) {
      const int c = idx / (P / 2), m2 = (idx % (P / 2)) * 2;
      const bool ok = (n0 + c) < lg.nlines;
      cp_async16(Xw + c * E::LDR + m2, x + (ok ? (n0 + c) * P + m2 : 0), ok);
    }
  } else {
    const bool fast = (lg.R % 8 == 0) && (n0 + 8 <= lg.nlines);
    if (fast) {
      const long long b0 = lg.base(n0);
#pragma unroll 4
      for (int idx = lane; idx < P * 4; idx += 32) {
        const int m = idx >> 2, c2 = (idx & 3) * 2;
        cp_async16(Xw + xaddr<P, false>(m, c2), x + b0 + (long long)m * lg.R + c2, true);
      }
    } else {
      const int c = lane & 7;
      const bool ok = (n0 + c) < lg.nlines;
      const long long bc = ok ? lg.base(n0 + c) : 0;
      for (int m = lane >> 3; m < P; m += 4) cp_async8(Xw + xaddr<P, false>(m, c), x + bc + (long long)m * lg.R, ok);
    }
  }
  cp_async_commit();
}


// Warp-level load of one 8-line block straight from the GLOBAL vector U (interior nodes only,
// lexicographic; elliptic.C:408-409) with the homogeneous-Dirichlet pad of MatMult_Elliptic
// (elliptic.C:305-308) applied on the fly: boundary nodes are zero-filled, so no padded copy of the
// field is ever materialised.  All extents equal P; `axis` is the chain axis, n0 the first line.
// NPART warps that share the block each load one NPART-th of it (warp `part`: lines c with c * NPART / 8 == part on the last
// axis, rows m with m / 4 % NPART == part otherwise).
template <int P, bool RIGHT, int NPART = 1>
__device__ __forceinline__ void load_block_from_U(double* Xw, const double* __restrict__ U, int d, int axis,
                                                  unsigned n0, int lane, const SlabGeom sg, int part = 0) {
  using E = EO<P>;
  // decode the d-1 digits (base P) of line n0 over the axes other than `axis`, fastest axis first;
  // the slowest digit is whatever remains (axis 0 may have a local extent != P in slab mode)
  unsigned rem = n0;
  long long gb = -sg.goff;  // global id of (line, m = 1) for c = 0, relative to the local vector
  long long ist = 1;        // interior stride of the axis being visited
  long long ist_a = 1, ist_fast = 1;
  int dig_fast = 0;
  bool inter = true;
  const int fast = RIGHT ? d - 2 : d - 1;
  const int slowest = axis == 0 ? 1 : 0;
  for (int j = d - 1; j >= 0; j--) {
    if (j == axis) {
      ist_a = ist;
    } else {
      int dig;
      if (j == slowest) {
        dig = (int)rem;
      } else {
        dig = (int)(rem % P);
        rem /= P;
      }
      const int lo = 1, hi = (j == 0 ? sg.n0g : P) - 2;
      const int gdig = dig + (j == 0 ? sg.i0 : 0);
      if (j == fast) {
        dig_fast = gdig;
        ist_fast = ist;
      } else {
        inter = inter && gdig >= lo && gdig <= hi;
      }
      gb += (long long)(gdig - 1) * ist;
    }
    ist *= (P - 2);
  }
  const int fast_hi = (fast == 0 ? sg.n0g : P) - 2;
  if (RIGHT) {
    // lanes run along the line (contiguous in U); 8 lines, ceil(P/32) passes each
    constexpr int PASSES = (P + 31) / 32;
    static_assert(8 % NPART == 0, "each part loads whole lines");
#pragma unroll 4
    for (int ip = 0; ip < 8 * PASSES / NPART; ip++) {
      const int i = part * (8 * PASSES / NPART) + ip;
      const int c = i / PASSES, m = lane + 32 * (i % PASSES);
      if (m >= P) continue;
      const bool ok = inter && (dig_fast + c >= 1) && (dig_fast + c <= fast_hi) && m >= 1 && m <= P - 2;
      cp_async8(Xw + c * E::LDR + m, U + (ok ? gb + c * ist_fast + (m - 1) : 0), ok);
    }
  } else {
    const int c = lane & 7;
    const bool okc = inter && (dig_fast + c >= 1) && (dig_fast + c <= fast_hi);
    const double* src = U + gb + c - ist_a;  // + m * ist_a  (ist_fast == 1 for the last axis)
#pragma unroll 4
    for (int m = (lane >> 3) + 4 * part; m < P; m += 4 * NPART) {
      const bool ok = okc && m >= 1 && m <= P - 2;
      cp_async8(Xw + xaddr<P, false>(m, c), ok ? src + (long long)m * ist_a : U, ok);
    }
  }
  cp_async_commit();
}

}  // namespace sb200
