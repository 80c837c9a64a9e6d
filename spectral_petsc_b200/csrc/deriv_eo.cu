// Even-odd persistent derivative kernel: y = D_axis x for ANY extent 2 <= P <= SB200_EO_MAX_P (the reference's ChebMult takes
// any extent, chebyshev.c:107-129), any (O, P, R) factorisation and any element stride / offset (the AoS velocity components of
// stokes.C:284-289,585,613), with the scatters and AXPY chains that surround a derivative in the reference fused in:
//   loader   : plain field | straight from the global (interior-only) vector with zero Dirichlet rows (VecScatter global -> local)
//   epilogue : y = D x | yin -+ D x | cropped into a global vector, optionally summed with the terms EARLIER jobs of the same launch
//              produced (the VecAXPY chain + VecScatter local -> global of stokes.C:584-592, 611-617, 668-673)
//
// Machinery (as in the fused chain kernels, chain.cuh): the two half-size matrices Ae / Bo of the centro-antisymmetric CGL matrix
// stay resident in shared memory (zero padded to HP = 8*MT rows, so odd P and P % 16 != 0 run the same DMMA tiles; the self-paired
// middle node of an odd P is folded into the matrices on the host, cheb_matrix.cpp), every warp owns an 8-line block, pulls tickets
// from a global counter and runs  load -> even-odd DMMA GEMM -> epilogue  with no CTA barrier after the matrix load.  Executed
// flops are half of the dense product that deriv_generic.cu performs.
#include "../../include/spectral_b200.h"
#include "chain.cuh"
#include "deriv.h"
#include "elliptic.h"

namespace sb200 {

namespace {

template <int MT>
struct EOG {
  static constexpr int HP = 8 * MT;   // padded pair count
  static constexpr int KS = HP / 4;   // k4 steps
  static constexpr int LDM = HP + 4;  // matrix leading dim in smem: (g*LDM + t) mod 16 distinct over a half-warp
  static constexpr int PP = 16 * MT;  // rows of a warp's block
  static constexpr int MAT_ELEMS = 2 * HP * LDM;
  static constexpr int BLOCK_ELEMS = PP * 8;
};

// Up to SB200_EO_MAX_JOBS derivatives that share the matrix run as ONE launch: the tickets of job j are [end[j-1], end[j]).
// (The reference applies D_0, D_1, D_2 back to back - stokes.C:584-590,611-614,639,668-671 - each on the full
// grid; one launch keeps every SM busy through the tail of each and loads Ae / Bo once.)
struct EoJob {
  const double* x;
  double* y;
  const double* yin;
  long long R, nlines;
  int xs, xoff, ys, yoff, mode;
  int vec;       // R % 8 == 0, unit strides, 16-byte aligned, plain loader and epilogue: the block's 8 lines are adjacent in memory
  unsigned end;  // exclusive prefix of item counts
  // fused scatters (see deriv.h)
  EoLineMap lm;
  const double* gsrc;
  int gs_stride, gs_off;
  double* gdst;
  int gd_stride, gd_off, fin, nterms, add, self_pos;
  int fvec;  // crop-sum with at most two terms whose fields hold the block's 8 lines adjacently (R % 8 == 0, unit stride, 16-byte aligned, no rhs)
  const double* term[SB200_EO_MAX_JOBS - 1];
  const double* sub;
  double sign;
  // pencil derivative of a slab partition: result rows go straight to their owners (see deriv.h)
  double* ypeer[SB200_MAX_RANKS];
  int peer_on, peer_nloc, peer_negate;
  long long peer_R, peer_col0;
};
struct EoParams {
  EoJob job[SB200_EO_MAX_JOBS];
  int njobs;
  int P;
  const double* Ae;
  const double* Bo;
  unsigned items;     // total
  unsigned wait_items;  // a job with terms reads them only after this many items (all of the earlier jobs') have finished
  int count_done;       // some job of this launch has terms: finished items are counted
  unsigned* sync;       // [0] ticket, [1] exited warps, [2] finished items
};

struct LineInfo {
  bool interior;   // every OTHER axis index of the line is interior
  long long gbase; // interior ordinal of the line's node at axis index 1 (the first interior node of the line)
  int comp;
};

__device__ __forceinline__ LineInfo decode_line(const EoLineMap& lm, unsigned n) {
  LineInfo li;
  li.comp = (int)(n % (unsigned)lm.nc);
  unsigned rem = n / (unsigned)lm.nc;
  li.interior = true;
  li.gbase = 0;
  for (int j = lm.d - 1; j >= 0; j--) {
    if (j == lm.axis) continue;
    const unsigned dj = (unsigned)lm.dim[j];
    const int ij = (int)(rem % dj);
    rem /= dj;
    li.interior = li.interior && ij >= 1 && ij <= (int)dj - 2;
    li.gbase += (long long)(ij - 1) * lm.istride[j];
  }
  return li;
}

template <int MT>
__device__ __forceinline__ void load_matrices_g(double* sm, const double* __restrict__ gAe, const double* __restrict__ gBo) {
  using E = EOG<MT>;
  for (int idx = threadIdx.x; idx < E::HP * E::HP / 2; idx += blockDim.x) {
    const int r = idx / (E::HP / 2), c2 = (idx % (E::HP / 2)) * 2;
    cp_async16(sm + r * E::LDM + c2, gAe + r * E::HP + c2, true);
    cp_async16(sm + E::HP * E::LDM + r * E::LDM + c2, gBo + r * E::HP + c2, true);
  }
  cp_async_commit();
}

__device__ __forceinline__ int xaddrL(int m, int c) { return m * 8 + (c ^ (((m >> 1) & 1) << 2)); }

// a[i], b[i] = Ae * s, Bo * d for the warp's 8 lines; acc[i][h] <-> pair index i*8+g, line 2t+h.  EXACT: P == 16*MT (no padded pairs).
template <int MT, bool EXACT>
__device__ __forceinline__ void eo_gemm_g(const double* __restrict__ Ae, const double* __restrict__ Bo, const double* __restrict__ Xw,
                                          double (&a)[MT][2], double (&b)[MT][2], int g, int t, int n, int hh) {
  using E = EOG<MT>;
#pragma unroll
  for (int i = 0; i < MT; i++) a[i][0] = a[i][1] = b[i][0] = b[i][1] = 0.0;
#pragma unroll 4
  for (int ks = 0; ks < E::KS; ks++) {
    const int kk = ks * 4 + t;
    double p = 0.0, q = 0.0;
    if (EXACT || kk < hh) {
      p = Xw[xaddrL(kk, g)];
      q = Xw[xaddrL(n - kk, g)];
    }
    const double s = p + q, d = p - q;
    double fa[MT], fb[MT];
#pragma unroll
    for (int i = 0; i < MT; i++) {
      fa[i] = Ae[(i * 8 + g) * E::LDM + kk];
      fb[i] = Bo[(i * 8 + g) * E::LDM + kk];
    }
#pragma unroll
    for (int i = 0; i < MT; i++) {
      dmma884(a[i][0], a[i][1], fa[i], s);
      dmma884(b[i][0], b[i][1], fb[i], d);
    }
  }
}

// FUSED = false compiles the plain derivative alone (no pad loader, no crop epilogue, no item counting): the launches of the large
// grids, whose inner loop must not share registers with the scatter code.
template <int MT, int NWARPS, bool EXACT, bool FUSED>
__global__ void __launch_bounds__(NWARPS * 32, 1) eo_deriv_kernel(EoParams q) {
  using E = EOG<MT>;
  extern __shared__ double sm[];
  double* Ae = sm;
  double* Bo = sm + E::HP * E::LDM;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int P = EXACT ? E::PP : q.P, n = P - 1, hh = (P + 1) >> 1;
  double* Xw = sm + E::MAT_ELEMS + warp * E::BLOCK_ELEMS;
  load_matrices_g<MT>(sm, q.Ae, q.Bo);

  auto grab = [&]() -> unsigned {
    unsigned tk = 0;
    if (lane == 0) tk = atomicAdd(q.sync, 1u);
    return __shfl_sync(0xffffffffu, tk, 0);
  };
  auto job_of = [&](unsigned tk) -> int {
    int j = 0;
    while (j + 1 < q.njobs && tk >= q.job[j].end) j++;
    return j;
  };
  auto line_base = [&](long long ln, long long R) -> long long {  // element index of (line ln, m = 0)
    const long long o = ln / R, r = ln - o * R;
    return o * (long long)P * R + r;
  };
  auto issue_load = [&](unsigned tk) {
    if (tk >= q.items) return;
    const int j = job_of(tk);
    const EoJob& p = q.job[j];
    const long long R = p.R;
    const long long n0 = (long long)(tk - (j ? q.job[j - 1].end : 0u)) * 8;
    if (FUSED && p.gsrc) {
      // fused pad: lane c = lane & 7 owns line n0 + c; boundary nodes (and lines beyond the end) are zero filled
      const int c = lane & 7;
      const bool ok = (n0 + c) < p.nlines;
      const LineInfo li = decode_line(p.lm, (unsigned)(ok ? n0 + c : 0));
      const bool inter = ok && li.interior;
      const long long ist = p.lm.istride[p.lm.axis];
      const double* src = p.gsrc + (li.gbase - ist) * p.gs_stride + p.gs_off + li.comp;  // + m * ist * gs_stride
      const long long step = ist * p.gs_stride;
#pragma unroll 4
      for (int m = lane >> 3; m < P; m += 4) {
        const bool v = inter && m >= 1 && m <= P - 2;
        cp_async8(Xw + xaddrL(m, c), v ? src + (long long)m * step : p.gsrc, v);
      }
    } else if (p.vec) {
      const long long b0 = line_base(n0, R);
#pragma unroll 4
      for (int idx = lane; idx < P * 4; idx += 32) {
        const int m = idx >> 2, c2 = (idx & 3) * 2;
        cp_async16(Xw + xaddrL(m, c2), p.x + b0 + (long long)m * R + c2, true);
      }
    } else {
      const int c = lane & 7;
      const bool ok = (n0 + c) < p.nlines;
      const long long bc = ok ? line_base(n0 + c, R) : 0;
#pragma unroll 4
      for (int m = lane >> 3; m < P; m += 4)
        cp_async8(Xw + xaddrL(m, c), p.x + (ok ? (bc + (long long)m * R) * p.xs + p.xoff : 0), ok);
    }
    cp_async_commit();
  };

  unsigned tk = grab();
  issue_load(tk);
  cp_async_wait<0>();
  __syncthreads();  // matrices visible to all warps

  while (tk < q.items) {
    const int j = job_of(tk);
    const EoJob& p = q.job[j];
    const long long R = p.R;
    const long long n0 = (long long)(tk - (j ? q.job[j - 1].end : 0u)) * 8;
    cp_async_wait<0>();
    __syncwarp();
    double a[MT][2], b[MT][2];
    eo_gemm_g<MT, EXACT>(Ae, Bo, Xw, a, b, g, t, n, hh);
    __syncwarp();  // block free: refill it while the epilogue drains
    const unsigned nxt = grab();
    issue_load(nxt);

    // thread-owned outputs: lines 2t, 2t+1; rows mt = i*8+g (a+b) and mb = n-mt (b-a); the middle row of an odd P is its own mirror
    if (FUSED && p.gdst) {
      if (p.nterms > 0) {
        // the terms are complete once every item of the earlier jobs has checked in
        if (lane == 0) {
          const long long t0 = clock64();
          while (*reinterpret_cast<volatile unsigned*>(q.sync + 2) < q.wait_items) {
            if (clock64() - t0 > (1ll << 33)) break;  // cannot happen (earlier tickets are held by running warps); never hang the GPU
          }
          __threadfence();
        }
        __syncwarp();
      }
      const long long ist = p.lm.istride[p.lm.axis];
      if (p.fvec) {
        // lines 2t, 2t+1 are adjacent in the term fields (R % 8 == 0): one 16-byte load per term and row serves both; every load
        // of a tile (top and mirrored row, all terms) is issued before the first use
        const long long l0 = n0 + 2 * t;
        const LineInfo li0 = decode_line(p.lm, (unsigned)l0), li1 = decode_line(p.lm, (unsigned)(l0 + 1));
        const long long lb = line_base(l0, R);
        double* __restrict__ dst0 = p.gdst + (li0.gbase - ist) * p.gd_stride + p.gd_off + li0.comp;
        double* __restrict__ dst1 = p.gdst + (li1.gbase - ist) * p.gd_stride + p.gd_off + li1.comp;
        const long long step = ist * p.gd_stride;
        const double* __restrict__ T0 = p.term[0];
        const double* __restrict__ T1 = p.term[1];
        const bool two = p.nterms == 2;
        if (li0.interior || li1.interior) {
#pragma unroll
          for (int i = 0; i < MT; i++) {
            const int mt = i * 8 + g, mb = n - mt;
            if (!EXACT && mt >= hh) continue;
            const bool lt = mt >= 1, lbm = (EXACT || mb != mt) && mb <= P - 2;  // (mt <= hh - 1 <= P - 2 and mb >= 1 always hold here)
            const long long et = lb + (long long)mt * R, eb = lb + (long long)mb * R;
            double2 t0t = make_double2(0.0, 0.0), t0b = t0t, t1t = t0t, t1b = t0t;
            if (lt) t0t = __ldcg(reinterpret_cast<const double2*>(T0 + et));
            if (lbm) t0b = __ldcg(reinterpret_cast<const double2*>(T0 + eb));
            if (two && lt) t1t = __ldcg(reinterpret_cast<const double2*>(T1 + et));
            if (two && lbm) t1b = __ldcg(reinterpret_cast<const double2*>(T1 + eb));
            const double vt[2] = {a[i][0] + b[i][0], a[i][1] + b[i][1]};
            const double vb[2] = {b[i][0] - a[i][0], b[i][1] - a[i][1]};
            const double s0t[2] = {t0t.x, t0t.y}, s0b[2] = {t0b.x, t0b.y}, s1t[2] = {t1t.x, t1t.y}, s1b[2] = {t1b.x, t1b.y};
#pragma unroll
            for (int h = 0; h < 2; h++) {
              if (!(h ? li1.interior : li0.interior)) continue;
              double* __restrict__ dst = h ? dst1 : dst0;
              // the chain in axis order: the job's own value enters at position self_pos
              double ct = 0.0, cb = 0.0;
              if (p.self_pos == 0) { ct = __dadd_rn(ct, __dmul_rn(p.sign, vt[h])); cb = __dadd_rn(cb, __dmul_rn(p.sign, vb[h])); }
              ct = __dadd_rn(ct, __dmul_rn(p.sign, s0t[h]));
              cb = __dadd_rn(cb, __dmul_rn(p.sign, s0b[h]));
              if (p.self_pos == 1) { ct = __dadd_rn(ct, __dmul_rn(p.sign, vt[h])); cb = __dadd_rn(cb, __dmul_rn(p.sign, vb[h])); }
              if (two) {
                ct = __dadd_rn(ct, __dmul_rn(p.sign, s1t[h]));
                cb = __dadd_rn(cb, __dmul_rn(p.sign, s1b[h]));
                if (p.self_pos == 2) { ct = __dadd_rn(ct, __dmul_rn(p.sign, vt[h])); cb = __dadd_rn(cb, __dmul_rn(p.sign, vb[h])); }
              }
              if (lt) dst[(long long)mt * step] = ct;
              if (lbm) dst[(long long)mb * step] = cb;
            }
          }
        }
      } else {
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const long long ln = n0 + 2 * t + h;
        if (ln >= p.nlines) continue;
        const LineInfo li = decode_line(p.lm, (unsigned)ln);
        if (!li.interior) continue;
        const long long lb = line_base(ln, R);
        double* __restrict__ dst = p.gdst + (li.gbase - ist) * p.gd_stride + p.gd_off + li.comp;  // + m * ist * gd_stride
        const double* __restrict__ sub = p.sub ? p.sub + (li.gbase - ist) * p.gd_stride + p.gd_off + li.comp : nullptr;
        const long long step = ist * p.gd_stride;
        // batches of thread-owned rows: every load of a batch is issued before the first use, so an item pays a few
        // L2 round trips instead of one per element
        constexpr int TB = MT >= 6 ? 2 : (MT < 4 ? MT : 4);  // tiles per batch (fewer where the accumulators leave few registers)
#pragma unroll
        for (int ib = 0; ib < MT; ib += TB) {
          constexpr int NB = TB * 2;
          int mrow[NB];
          double val[NB], acc[NB];
          bool live[NB];
#pragma unroll
          for (int ii = 0; ii < NB / 2; ii++) {
            const int i = ib + ii;
            const int mt = i < MT ? i * 8 + g : P, mb = n - mt;  // (i >= MT only when MT % TB != 0: dead slots)
            const bool tv = i < MT && (EXACT || mt < hh);
            mrow[2 * ii] = mt;
            mrow[2 * ii + 1] = mb;
            live[2 * ii] = tv && mt >= 1 && mt <= P - 2;
            live[2 * ii + 1] = tv && (EXACT || mb != mt) && mb >= 1 && mb <= P - 2;
            val[2 * ii] = i < MT ? a[i < MT ? i : 0][h] + b[i < MT ? i : 0][h] : 0.0;
            val[2 * ii + 1] = i < MT ? b[i < MT ? i : 0][h] - a[i < MT ? i : 0][h] : 0.0;
          }
          if (p.fin == EO_FIN_SUM) {
#pragma unroll
            for (int k = 0; k < NB; k++) acc[k] = 0.0;
            for (int tt = 0; tt <= p.nterms; tt++) {
              if (tt == p.self_pos) {
#pragma unroll
                for (int k = 0; k < NB; k++) acc[k] = __dadd_rn(acc[k], __dmul_rn(p.sign, val[k]));
              }
              if (tt == p.nterms) break;
              const double* __restrict__ T = p.term[tt];
              double tv[NB];
#pragma unroll
              for (int k = 0; k < NB; k++) tv[k] = live[k] ? __ldcg(T + (lb + (long long)mrow[k] * R) * p.ys + p.yoff) : 0.0;
#pragma unroll
              for (int k = 0; k < NB; k++) acc[k] = __dadd_rn(acc[k], __dmul_rn(p.sign, tv[k]));
            }
          } else {
#pragma unroll
            for (int k = 0; k < NB; k++) acc[k] = val[k];
            if (p.add) {
              double dv[NB];
#pragma unroll
              for (int k = 0; k < NB; k++) dv[k] = live[k] ? dst[(long long)mrow[k] * step] : 0.0;
#pragma unroll
              for (int k = 0; k < NB; k++) acc[k] = dv[k] + acc[k];
            }
          }
          if (sub) {
            double sv[NB];
#pragma unroll
            for (int k = 0; k < NB; k++) sv[k] = live[k] ? sub[(long long)mrow[k] * step] : 0.0;
#pragma unroll
            for (int k = 0; k < NB; k++) acc[k] = acc[k] + (-1.0) * sv[k];
          }
#pragma unroll
          for (int k = 0; k < NB; k++)
            if (live[k]) dst[(long long)mrow[k] * step] = acc[k];
        }
      }
      }
    } else if (FUSED && p.peer_on) {
      // O == 1, unit strides, R % 8 == 0: columns n0 + 2t, +1 of row m -> the owner of plane m (16-byte peer stores)
      const long long col = p.peer_col0 + n0 + 2 * t;
#pragma unroll
      for (int i = 0; i < MT; i++) {
        const int mt = i * 8 + g, mb = n - mt;
        if (!EXACT && mt >= hh) continue;
        const int qt = mt / p.peer_nloc, qb = mb / p.peer_nloc;
        double2 vt = make_double2(a[i][0] + b[i][0], a[i][1] + b[i][1]);
        double2 vb = make_double2(b[i][0] - a[i][0], b[i][1] - a[i][1]);
        if (p.peer_negate) {
          vt = make_double2(0.0 - vt.x, 0.0 - vt.y);
          vb = make_double2(0.0 - vb.x, 0.0 - vb.y);
        }
        st2(p.ypeer[qt] + (long long)(mt - qt * p.peer_nloc) * p.peer_R + col, vt.x, vt.y);
        if (EXACT || mb != mt) st2(p.ypeer[qb] + (long long)(mb - qb * p.peer_nloc) * p.peer_R + col, vb.x, vb.y);
      }
    } else if (p.vec) {
      const long long base = line_base(n0, R) + 2 * t;
#pragma unroll
      for (int i = 0; i < MT; i++) {
        const int mt = i * 8 + g, mb = n - mt;
        if (!EXACT && mt >= hh) continue;
        const long long et = base + (long long)mt * R, eb = base + (long long)mb * R;
        double2 vt = make_double2(a[i][0] + b[i][0], a[i][1] + b[i][1]);
        double2 vb = make_double2(b[i][0] - a[i][0], b[i][1] - a[i][1]);
        if (p.mode != DERIV_STORE) {
          const double2 yt = p.yin ? ld2(p.yin + et) : make_double2(0.0, 0.0);
          const double2 yb = p.yin ? ld2(p.yin + eb) : make_double2(0.0, 0.0);
          if (p.mode == DERIV_SUB) {
            vt = make_double2(yt.x - vt.x, yt.y - vt.y);
            vb = make_double2(yb.x - vb.x, yb.y - vb.y);
          } else {
            vt = make_double2(yt.x + vt.x, yt.y + vt.y);
            vb = make_double2(yb.x + vb.x, yb.y + vb.y);
          }
        }
        st2(p.y + et, vt.x, vt.y);
        if (EXACT || mb != mt) st2(p.y + eb, vb.x, vb.y);
      }
    } else {
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const long long ln = n0 + 2 * t + h;
        if (ln >= p.nlines) continue;
        const long long lb = line_base(ln, R);
#pragma unroll
        for (int i = 0; i < MT; i++) {
          const int mt = i * 8 + g, mb = n - mt;
          if (!EXACT && mt >= hh) continue;
          const long long et = (lb + (long long)mt * R) * p.ys + p.yoff;
          const long long eb = (lb + (long long)mb * R) * p.ys + p.yoff;
          double vt = a[i][h] + b[i][h], vb = b[i][h] - a[i][h];
          if (p.mode == DERIV_SUB) {
            vt = (p.yin ? p.yin[et] : 0.0) - vt;
            vb = (p.yin ? p.yin[eb] : 0.0) - vb;
          } else if (p.mode == DERIV_ADD) {
            vt = (p.yin ? p.yin[et] : 0.0) + vt;
            vb = (p.yin ? p.yin[eb] : 0.0) + vb;
          }
          p.y[et] = vt;
          if (EXACT || mb != mt) p.y[eb] = vb;
        }
      }
    }
    if (FUSED && q.count_done && !(p.gdst && p.nterms > 0)) {
      // this item's term rows are visible device-wide before it checks in
      __threadfence();
      __syncwarp();
      if (lane == 0) atomicAdd(q.sync + 2, 1u);
    }
    tk = nxt;
  }
  cp_async_wait<0>();
  if (lane == 0) {
    const unsigned gone = atomicAdd(q.sync + 1, 1u);
    if (gone == gridDim.x * NWARPS - 1) {  // the last warp to leave re-arms the counters
      q.sync[0] = 0;
      q.sync[1] = 0;
      q.sync[2] = 0;
    }
  }
}

template <int MT, int NWARPS, bool EXACT, bool FUSED>
int launch_eo(const EoParams& q, cudaStream_t s) {
  using E = EOG<MT>;
  auto kern = eo_deriv_kernel<MT, NWARPS, EXACT, FUSED>;
  const size_t smem = (size_t)(E::MAT_ELEMS + NWARPS * E::BLOCK_ELEMS) * sizeof(double);
  // the opt-in above 48 KB is per device: remembered per device (a small grid's launch costs more on the host than on the GPU)
  static bool attr[64] = {};
  static int nsm[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  const int di = dev & 63;
  if (!attr[di]) {
    SB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int v = 148;
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    nsm[di] = v;
    attr[di] = true;
  }
  const int sms = nsm[di];
  long long grid = (q.items + NWARPS - 1) / NWARPS;
  if (grid > sms) grid = sms;
  if (grid < 1) grid = 1;
  kern<<<(unsigned)grid, NWARPS * 32, smem, s>>>(q);
  count_launch();
  SB_CUDA(cudaGetLastError());
  return 0;
}

template <int MT, int NWARPS>
int launch_mt(const EoParams& q, cudaStream_t s) {
  bool fused = false;
  for (int j = 0; j < q.njobs; j++) fused = fused || q.job[j].gsrc || q.job[j].gdst || q.job[j].peer_on;
  if (q.P == 16 * MT) return fused ? launch_eo<MT, NWARPS, true, true>(q, s) : launch_eo<MT, NWARPS, true, false>(q, s);
  return fused ? launch_eo<MT, NWARPS, false, true>(q, s) : launch_eo<MT, NWARPS, false, false>(q, s);
}

}  // namespace

bool deriv_eo_supported(const DerivParams& p) {
  if (!p.Ae || !p.Bo || p.npeer > 1) return false;
  return p.P >= 2 && p.P <= SB200_EO_MAX_P && p.HP >= (p.P + 1) / 2 && p.HP % 8 == 0 && p.HP <= 80;
}

int deriv_eo_batch(const DerivParams* jobs, int n, unsigned* sync, cudaStream_t s) {
  SB_CHECK(n >= 1 && n <= SB200_EO_MAX_JOBS, SB200_ERR_USER, "even-odd derivative: bad job count");
  EoParams q;
  q.njobs = n;
  q.P = jobs[0].P;
  q.Ae = jobs[0].Ae;
  q.Bo = jobs[0].Bo;
  q.sync = sync;
  q.wait_items = 0;
  q.count_done = 0;
  unsigned total = 0;
  for (int j = 0; j < n; j++) {
    const DerivParams& p = jobs[j];
    SB_CHECK(deriv_eo_supported(p) && p.P == jobs[0].P && p.Ae == q.Ae, SB200_ERR_USER, "even-odd derivative: jobs must share the matrix");
    SB_CHECK(p.gsrc || p.gdst || p.inplace_ok || p.peer_on || p.x != p.y, SB200_ERR_ARG, "deriv: x and y must not alias (chebyshev.c:127)");
    SB_CHECK((!p.gsrc && !p.gdst) || (p.lm.d >= 1 && p.lm.d <= SB200_EO_MAX_JOBS && p.lm.nc >= 1), SB200_ERR_USER, "even-odd derivative: fused scatter without a line map");
    EoJob& e = q.job[j];
    e.x = p.x;
    e.y = p.y;
    e.yin = p.yin;
    e.R = p.R;
    e.nlines = p.O * p.R;
    e.xs = p.xs;
    e.xoff = p.xoff;
    e.ys = p.ys;
    e.yoff = p.yoff;
    e.mode = p.mode;
    e.lm = p.lm;
    e.gsrc = p.gsrc;
    e.gs_stride = p.gs_stride;
    e.gs_off = p.gs_off;
    e.gdst = p.gdst;
    e.gd_stride = p.gd_stride;
    e.gd_off = p.gd_off;
    e.fin = p.gdst ? p.fin : EO_FIN_NONE;
    e.nterms = (p.gdst && p.fin == EO_FIN_SUM) ? p.nterms : 0;
    e.add = p.add;
    for (int t = 0; t < SB200_EO_MAX_JOBS - 1; t++) e.term[t] = p.term[t];
    e.sub = p.sub;
    e.sign = p.sign;
    for (int r = 0; r < SB200_MAX_RANKS; r++) e.ypeer[r] = p.ypeer[r];
    e.peer_on = p.peer_on;
    e.peer_nloc = p.peer_nloc;
    e.peer_negate = p.peer_negate;
    e.peer_R = p.peer_R;
    e.peer_col0 = p.peer_col0;
    SB_CHECK(!p.peer_on || (!p.gdst && p.O == 1 && p.R % 8 == 0 && p.xs == 1 && p.peer_nloc >= 1 && p.peer_R % 2 == 0 && p.peer_col0 % 2 == 0), SB200_ERR_USER,
             "even-odd derivative: the peer epilogue needs a unit-stride pencil with an even column range");
    e.self_pos = (p.gdst && p.fin == EO_FIN_SUM) ? (p.self_pos < 0 ? e.nterms : p.self_pos) : 0;
    SB_CHECK(e.self_pos >= 0 && e.self_pos <= e.nterms, SB200_ERR_USER, "even-odd derivative: bad chain position");
    e.fvec = p.gdst && p.fin == EO_FIN_SUM && e.nterms >= 1 && e.nterms <= 2 && !p.sub && (p.R % 8 == 0) && p.ys == 1 && p.yoff == 0 &&
             ((reinterpret_cast<uintptr_t>(p.term[0]) | reinterpret_cast<uintptr_t>(e.nterms == 2 ? p.term[1] : nullptr)) % 16 == 0);
    SB_CHECK(e.nterms >= 0 && e.nterms < SB200_EO_MAX_JOBS, SB200_ERR_USER, "even-odd derivative: too many terms");
    SB_CHECK(!p.gdst || p.fin == EO_FIN_SUM || p.fin == EO_FIN_RAW, SB200_ERR_USER, "even-odd derivative: bad crop mode");
    if (e.nterms > 0) {
      // every earlier job must be a plain producer; they all finish before the first reader proceeds
      if (!q.count_done) q.wait_items = total;
      q.count_done = 1;
    }
    e.vec = !p.gsrc && !p.gdst && (p.R % 8 == 0) && p.xs == 1 && (p.peer_on || (p.ys == 1 && p.yoff == 0)) && p.xoff == 0 &&
            ((reinterpret_cast<uintptr_t>(p.x) | reinterpret_cast<uintptr_t>(p.peer_on ? nullptr : p.y) | reinterpret_cast<uintptr_t>(p.yin)) % 16 == 0);
    SB_CHECK(!p.peer_on || e.vec, SB200_ERR_USER, "even-odd derivative: the peer epilogue needs the 16-byte block loader (aligned pencil)");
    total += (unsigned)((e.nlines + 7) / 8);
    e.end = total;
  }
  q.items = total;
  switch (jobs[0].HP / 8) {
    case 1: return launch_mt<1, 16>(q, s);
    case 2: return launch_mt<2, 16>(q, s);
    case 3: return launch_mt<3, 16>(q, s);
    case 4: return launch_mt<4, 16>(q, s);
    case 5: return launch_mt<5, 16>(q, s);
    case 6: return launch_mt<6, 16>(q, s);
    case 7: return launch_mt<7, 16>(q, s);
    case 8: return launch_mt<8, 16>(q, s);
    case 9: return launch_mt<9, 12>(q, s);
    case 10: return launch_mt<10, 10>(q, s);
  }
  set_last_error("even-odd derivative: unsupported extent");
  return SB200_ERR_SUP;
}

int deriv_eo_jobs(const DerivParams* jobs, int n, unsigned* sync, cudaStream_t s) {
  bool same = true;
  for (int k = 1; k < n; k++) same = same && jobs[k].Ae == jobs[0].Ae && jobs[k].P == jobs[0].P;
  if (same) return deriv_eo_batch(jobs, n, sync, s);
  for (int k = 0; k < n; k++) SB_TRY(deriv_eo_batch(jobs + k, 1, sync, s));
  return 0;
}

int deriv_eo_apply(const DerivParams& p, unsigned* sync, cudaStream_t s) { return deriv_eo_batch(&p, 1, sync, s); }

}  // namespace sb200
