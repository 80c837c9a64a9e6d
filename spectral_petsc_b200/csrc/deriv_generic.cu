// Generic per-axis Chebyshev derivative: y = D_axis x for a row-major array factored as
// (O, P, R) around the differentiated axis (replaces ChebMult, chebyshev.c:142-199, for any rank,
// any axis and any extent, including the AoS velocity layout of stokes.C:284-289).
//
// The derivative is the dense P x P CGL matrix applied as a batched GEMM on the FP64 tensor
// pipe (mma.sync m8n8k4 f64 -> DMMA.8x8x4):   C[i][n] = sum_k D[i][k] * X[k][n]
// where a "column" n is one grid line.  Two staging layouts keep global loads coalesced:
//   LEFT  (R large): columns of one o-slab are contiguous in r  -> B tile stored [k][n]
//   RIGHT (R small): a line's k-run is (nearly) contiguous       -> B tile stored [n][k]
// D (zero padded to a multiple of 32) streams through shared memory in K-chunks of 32 with a
// 2-stage cp.async pipeline.  Epilogue modes implement the reference's VecAXPY accumulation
// (elliptic.C:331-334, stokes.C:590,671) without an extra pass.
#include "deriv.h"

#include "common.cuh"
#include "../../include/spectral_b200.h"

namespace sb200 {

namespace {

constexpr int KC = 32;        // K chunk
constexpr int LDK = KC + 4;   // padded leading dim for [row][k] tiles: (4g + t) mod 16 distinct
constexpr int NTHREADS = 256;

template <int TM, int TN, bool LEFT>
struct TileCfg {
  static constexpr int LDB = LEFT ? (TN + 4) : LDK;
  static constexpr int A_ELEMS = TM * LDK;
  static constexpr int B_ELEMS = LEFT ? (KC * LDB) : (TN * LDK);
  static constexpr int STAGE_ELEMS = A_ELEMS + B_ELEMS;
  static constexpr size_t SMEM_BYTES = 2 * (size_t)STAGE_ELEMS * sizeof(double);
};

template <int TM, int WM, int WN, bool LEFT>
__global__ void __launch_bounds__(NTHREADS) deriv_kernel(DerivParams p) {
  constexpr int TN = WN * 32;
  constexpr int MT = TM / WM / 8;
  constexpr int NT = 4;
  using Cfg = TileCfg<TM, TN, LEFT>;
  extern __shared__ double smem[];

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const int wm0 = (warp / WN) * (TM / WM);
  const int wn0 = (warp % WN) * 32;
  const int m0 = blockIdx.z * TM;
  const bool slab = p.npeer > 1;
  const int mout = slab ? p.nloc : p.P;  // output rows this launch produces

  // Column bookkeeping.
  const long long R = p.R;
  const long long PR = (long long)p.P * R;
  long long o_base;      // LEFT: the slab o; RIGHT: first o-group of this tile
  long long r_base = 0;  // LEFT: first column r of this tile
  int ncols;             // valid columns in this tile
  int groups = 1;        // RIGHT: o-groups per tile
  if (LEFT) {
    const long long ntiles = (R + TN - 1) / TN;
    o_base = blockIdx.x / ntiles;
    r_base = (long long)(blockIdx.x % ntiles) * TN;
    long long rem = R - r_base;
    ncols = rem < TN ? (int)rem : TN;
  } else {
    groups = TN / (int)R;
    o_base = (long long)blockIdx.x * groups;
    long long rem = p.O - o_base;
    if (rem < groups) groups = (int)rem;
    ncols = groups * (int)R;
  }

  auto load_stage = [&](int stage, int k0) {
    double* As = smem + stage * Cfg::STAGE_ELEMS;
    double* Bs = As + Cfg::A_ELEMS;
    // A tile: D[m0 + m][k0 + k], 16-byte copies (D is padded: Pp % 32 == 0, rows 16B aligned).
    for (int idx = tid; idx < TM * (KC / 2); idx += NTHREADS) {
      int m = idx / (KC / 2), k2 = (idx % (KC / 2)) * 2;
      bool ok = (m0 + m) < (slab ? mout : p.Pp);
      const double* src = p.D + (size_t)(ok ? (p.row0 + m0 + m) : 0) * p.Pp + k0 + k2;
      cp_async16(As + m * LDK + k2, src, ok);
    }
    if (LEFT) {
      for (int idx = tid; idx < KC * TN; idx += NTHREADS) {
        int k = idx / TN, n = idx % TN;
        bool ok = (k0 + k) < p.P && n < ncols;
        const double* xo = p.x;
        long long e;
        if (slab) {
          const int kg = ok ? k0 + k : 0, q = kg / p.nloc;
          xo = p.xpeer[q];
          e = (long long)(kg - q * p.nloc) * R + r_base + n;
        } else {
          e = o_base * PR + (long long)(k0 + k) * R + r_base + n;
        }
        cp_async8(Bs + k * Cfg::LDB + n, xo + (ok ? e * p.xs + p.xoff : 0), ok);
      }
    } else {
      // per o-group the chunk k in [k0,k0+KC), r in [0,R) is contiguous: KC*R elements
      const int per = KC * (int)R;
      for (int idx = tid; idx < groups * per; idx += NTHREADS) {
        int og = idx / per, w = idx % per;
        int k = w / (int)R, r = w % (int)R;
        bool ok = (k0 + k) < p.P;
        long long e = (o_base + og) * PR + (long long)(k0 + k) * R + r;
        cp_async8(Bs + (og * (int)R + r) * LDK + k, p.x + (ok ? e * p.xs + p.xoff : 0), ok);
      }
      // zero the unused column slots once per stage so stale data never turns into NaNs
      for (int idx = tid + ncols * KC; idx < TN * KC; idx += NTHREADS) {
        int n = idx / KC, k = idx % KC;
        Bs[n * LDK + k] = 0.0;
      }
    }
    cp_async_commit();
  };

  double acc[MT][NT][2];
#pragma unroll
  for (int i = 0; i < MT; i++)
#pragma unroll
    for (int j = 0; j < NT; j++) acc[i][j][0] = acc[i][j][1] = 0.0;

  const int nk = p.Pp / KC;
  load_stage(0, 0);
  for (int kc = 0; kc < nk; kc++) {
    if (kc + 1 < nk) {
      load_stage((kc + 1) & 1, (kc + 1) * KC);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const double* As = smem + (kc & 1) * Cfg::STAGE_ELEMS;
    const double* Bs = As + Cfg::A_ELEMS;
#pragma unroll
    for (int ks = 0; ks < KC / 4; ks++) {
      double a[MT], b[NT];
#pragma unroll
      for (int i = 0; i < MT; i++) a[i] = As[(wm0 + i * 8 + g) * LDK + ks * 4 + t];
#pragma unroll
      for (int j = 0; j < NT; j++) {
        if (LEFT)
          b[j] = Bs[(ks * 4 + t) * Cfg::LDB + wn0 + j * 8 + g];
        else
          b[j] = Bs[(wn0 + j * 8 + g) * LDK + ks * 4 + t];
      }
#pragma unroll
      for (int i = 0; i < MT; i++)
#pragma unroll
        for (int j = 0; j < NT; j++) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
    }
    __syncthreads();
  }

  // Epilogue.
#pragma unroll
  for (int i = 0; i < MT; i++) {
    const int row = m0 + wm0 + i * 8 + g;
    if (row >= mout) continue;
#pragma unroll
    for (int j = 0; j < NT; j++) {
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const int n = wn0 + j * 8 + 2 * t + h;
        if (n >= ncols) continue;
        long long e;
        if (LEFT) {
          e = o_base * PR + (long long)row * R + r_base + n;
        } else {
          int og = n / (int)R, r = n % (int)R;
          e = (o_base + og) * PR + (long long)row * R + r;
        }
        const long long ye = e * p.ys + p.yoff;
        double v = acc[i][j][h];
        if (p.mode == DERIV_SUB) {
          v = (p.yin ? p.yin[ye] : 0.0) - v;
        } else if (p.mode == DERIV_ADD) {
          v = (p.yin ? p.yin[ye] : 0.0) + v;
        }
        p.y[ye] = v;
      }
    }
  }
}

template <int TM, int WM, int WN, bool LEFT>
int launch_cfg(const DerivParams& p, cudaStream_t stream) {
  constexpr int TN = WN * 32;
  using Cfg = TileCfg<TM, TN, LEFT>;
  static bool attr_set[64] = {};  // the opt-in above 48 KB of dynamic shared memory is per device
  auto kern = deriv_kernel<TM, WM, WN, LEFT>;
  int cur_dev = 0;
  cudaGetDevice(&cur_dev);
  if (!attr_set[cur_dev & 63]) {
    SB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM_BYTES));
    attr_set[cur_dev & 63] = true;
  }
  dim3 grid;
  if (LEFT) {
    const long long nb = ((p.R + TN - 1) / TN) * p.O;
    SB_CHECK(nb < (1ll << 31), SB200_ERR_SUP, "deriv: grid too large");
    const int mout = p.npeer > 1 ? p.nloc : p.P;
    grid = dim3((unsigned)nb, 1, (unsigned)((mout + TM - 1) / TM));
  } else {
    int groups = TN / (int)p.R;
    grid = dim3((unsigned)((p.O + groups - 1) / groups), 1, (unsigned)((p.P + TM - 1) / TM));
  }
  kern<<<grid, NTHREADS, Cfg::SMEM_BYTES, stream>>>(p);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return 0;
}

template <bool LEFT>
int launch_by_P(const DerivParams& p, cudaStream_t stream) {
  const int rows = p.npeer > 1 ? p.nloc : p.P;  // the row tile follows the rows this rank produces
  if (rows <= 16) return launch_cfg<16, 1, 8, LEFT>(p, stream);
  if (rows <= 32) return launch_cfg<32, 1, 8, LEFT>(p, stream);
  if (rows <= 64) return launch_cfg<64, 2, 4, LEFT>(p, stream);
  return launch_cfg<128, 4, 2, LEFT>(p, stream);
}

}  // namespace

int deriv_apply(const DerivParams& p, cudaStream_t stream) {
  SB_CHECK(p.P >= 2 && p.O >= 1 && p.R >= 1, SB200_ERR_USER, "deriv: bad extents");
  SB_CHECK(p.x != p.y, SB200_ERR_ARG, "deriv: x and y must not alias (chebyshev.c:127)");
  if (p.sync && deriv_eo_supported(p)) return deriv_eo_apply(p, p.sync, stream);
  if (p.npeer > 1) {
    SB_CHECK(p.O == 1 && p.nloc >= 1 && p.nloc * p.npeer == p.P, SB200_ERR_USER, "deriv: bad slab partition");
    return launch_by_P<true>(p, stream);
  }
  // LEFT needs enough contiguous columns per slab to fill a tile; otherwise batch o-groups.
  const int tn = p.P <= 32 ? 256 : (p.P <= 64 ? 128 : 64);
  if (p.R >= tn / 2) return launch_by_P<true>(p, stream);
  return launch_by_P<false>(p, stream);
}

}  // namespace sb200
