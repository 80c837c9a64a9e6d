// Single-launch persistent MatMult_Elliptic (elliptic.C:297-339) for grids with all extents equal to
// P (P % 16 == 0):  ONE kernel runs the chains of every axis.
//
// Work item = (axis k, block of 8*NT grid lines of that axis); items are handed out in order through a
// global ticket counter, all axes but the last first.  A warp owns its item end to end (chain.cuh):
//     load w block -> GEMM1 (even-odd DMMA) -> flux in registers -> in-place -> GEMM2 -> epilogue.
// Non-last axes store their term  D_k f_k  into a partial field (phase A launch); the last axis
// (R == 1, phase B launch) finishes   V = crop(((0 - p_0) - p_1 ...) - D_l f_l),  i.e. exactly the
// reference's accumulation order (elliptic.C:331-334).  Phase B is a programmatic dependent launch:
// its CTAs start on SMs as phase A drains, run GEMM1/flux/GEMM2 of their first items, and only block
// (griddepcontrol.wait) right before they read the partials.  Because every warp pulls several items
// of different phase, the global-memory phases of some warps overlap the tensor phases of the others.
#include <cstdlib>

#include "../../include/spectral_b200.h"
#include "chain.cuh"
#include "deriv.h"
#include "elliptic.h"
#include "persist.h"

// Ablation / timeline switches exist only in diagnostic builds (make ablate: -DSB200_ABLATE -> libspectral_b200_ablate.so);
// the production library compiles every XF() to false and never reads SB200_XFLAGS.
#ifdef SB200_ABLATE
#define XF(p, bit) (((p).xflags & (bit)) != 0)
#else
#define XF(p, bit) false
#endif

#ifdef SB200_TRACE
#define STAMP(k) do { if (lane == 0 && p.trace) tr[k] = clock64(); } while (0)
#else
#define STAMP(k) do { } while (0)
#endif

namespace sb200 {

namespace {

// Debug timeline (xflags & 64): global-timer stamps of the slab step's milestones, kept behind the
// counters in the sync block ((unsigned long long*)sync + 16 ...): even slots take a minimum, odd a maximum.
__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void tl_stamp(const PersistParams& p, int slot) {
  if (!XF(p, 64) || p.epoch != p.tl_epoch) return;
  unsigned long long* ts = reinterpret_cast<unsigned long long*>(p.sync) + 16;
  const unsigned long long t = gtime();
  atomicMin(ts + 2 * slot, t);
  atomicMax(ts + 2 * slot + 1, t);
}


template <int P, int NT, bool RIGHT, int MW = 1>
__device__ __forceinline__ void load_item(double* Xw, const double* __restrict__ U, int d, int axis,
                                          long long n0, int lane, const SlabGeom sg, int part = 0) {
  constexpr int BE = RIGHT ? EO<P>::BLOCK_ELEMS_RIGHT : EO<P>::BLOCK_ELEMS_LEFT;
#pragma unroll
  for (int j = 0; j < NT; j++) load_block_from_U<P, RIGHT, MW>(Xw + j * BE, U, d, axis, (unsigned)(n0 + 8 * j), lane, sg, part);
}

// MW == 2: the two warps of a pair (warps 2q, 2q+1 of the CTA) share one item and meet at named barrier 1 + q
// (barrier 0 is __syncthreads); MW == 1: the item is warp-private.
template <int MW>
__device__ __forceinline__ void item_sync() {
  if (MW == 1) {
    __syncwarp();
  } else {
    asm volatile("bar.sync %0, 64;" ::"r"(1 + (int)(threadIdx.x >> 6)) : "memory");
  }
}

// Flux operands of two tiles (top and bottom pair each): eta, deta, gradu.
struct FluxBuf {
  double2 e[2][2], de[2][2], gg[2][2];
};

template <int P, bool RIGHT, int TN>
__device__ __forceinline__ void flux_load(FluxBuf& f, const Own<P, RIGHT>& own, int ib, const double* __restrict__ eta,
                                          const double* __restrict__ deta, const double* __restrict__ g0) {
#pragma unroll
  for (int ii = 0; ii < 2; ii++) {
    if (ib + ii >= TN) continue;  // (odd TN: the last pair of tiles is a single tile)
    if (eta == nullptr) {
      f.e[ii][0] = f.e[ii][1] = make_double2(1.5, 1.5);
      f.de[ii][0] = f.de[ii][1] = f.gg[ii][0] = f.gg[ii][1] = make_double2(0.25, 0.25);
      continue;
    }
    const long long ot = own.top(ib + ii), ob = own.bot(ib + ii);
    f.e[ii][0] = ldg2(eta + ot);
    f.e[ii][1] = ldg2(eta + ob);
    f.de[ii][0] = ldg2(deta + ot);
    f.de[ii][1] = ldg2(deta + ob);
    f.gg[ii][0] = ldg2(g0 + ot);
    f.gg[ii][1] = ldg2(g0 + ob);
  }
}

// elliptic.C:319-323 for tiles ib, ib+1:  f = eta*y + (deta*w)*g0, written over w in the block.
template <int P, bool RIGHT, int TN>
__device__ __forceinline__ void flux_apply(const FluxBuf& f, const Own<P, RIGHT>& own, int ib, double* Xj,
                                           const double (&a)[TN][2], const double (&b)[TN][2]) {
#pragma unroll
  for (int ii = 0; ii < 2; ii++) {
    const int i = ib + ii;
    if (i >= TN) continue;
    const int st = own.stop(i), sb = own.sbot(i);
    const double2 wt = ld2(Xj + st), wb = ld2(Xj + sb);
    const double yt0 = a[i][0] + b[i][0], yt1 = a[i][1] + b[i][1];
    const double yb0 = RIGHT ? b[i][1] - a[i][1] : b[i][0] - a[i][0];
    const double yb1 = RIGHT ? b[i][0] - a[i][0] : b[i][1] - a[i][1];
    const double ft0 = __dadd_rn(__dmul_rn(f.e[ii][0].x, yt0), __dmul_rn(__dmul_rn(f.de[ii][0].x, wt.x), f.gg[ii][0].x));
    const double ft1 = __dadd_rn(__dmul_rn(f.e[ii][0].y, yt1), __dmul_rn(__dmul_rn(f.de[ii][0].y, wt.y), f.gg[ii][0].y));
    const double fb0 = __dadd_rn(__dmul_rn(f.e[ii][1].x, yb0), __dmul_rn(__dmul_rn(f.de[ii][1].x, wb.x), f.gg[ii][1].x));
    const double fb1 = __dadd_rn(__dmul_rn(f.e[ii][1].y, yb1), __dmul_rn(__dmul_rn(f.de[ii][1].y, wb.y), f.gg[ii][1].y));
    st2(Xj + st, ft0, ft1);
    st2(Xj + sb, fb0, fb1);
  }
}

// The whole chain for one item.  Returns after the epilogue stores are issued.
// DEEP: keep one flux batch in flight across GEMM1 and double-buffer the batches (needs registers).
// PENCIL (slab mode, axis 0): n0 is the line index inside this rank's pencil; the flux operands come
// from the pencil-layout state and the result rows are pushed to the part[0] array of the planes' owners.
// WAITDONE (slab mode, last axis, same launch as the local axes): their partials are complete once every local item has checked in,
// part[0] once every rank has raised its DONE flag.
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, int c0, int c1, const void* smem_src) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem_src);
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(map), "r"(c0), "r"(c1), "r"(s) : "memory");
}

struct NoEarly {
  __device__ __forceinline__ void operator()(int) const {}
};

// refill(0) runs right before the second GEMM, refill(1) right after it, refill(2) once every warp of the item has left it (the block is
// free): the single-GPU kernel takes its next ticket around GEMM2 and issues that item's load at refill(2), so the load flies during
// the epilogue instead of after it.
// MW warps share the item: warp h of them owns pair tiles [h * MT / MW, (h + 1) * MT / MW) - GEMM rows, flux and epilogue - and all
// of them read the whole block for the B fragments.
template <int P, int NT, bool RIGHT, bool DEEP, int MW = 1, bool PENCIL = false, bool WAITDONE = false, typename F = NoEarly>
__device__ __forceinline__ void run_item(const PersistParams& p, int axis, long long n0, const double* Ae,
                                         const double* Bo, double* Xw, int lane, const SlabMaps* maps = nullptr, double* stage = nullptr,
                                         F refill = F()) {
  using E = EO<P>;
  static_assert(!(PENCIL && RIGHT), "pencil items are strided-axis items");
  static_assert(E::MT % MW == 0 && (MW == 1 || (NT == 1 && DEEP && !PENCIL && !WAITDONE)), "split items: single-GPU, one block");
  constexpr int BE = RIGHT ? E::BLOCK_ELEMS_RIGHT : E::BLOCK_ELEMS_LEFT;
  constexpr int TN = E::MT / MW;  // pair tiles of this warp
  const int h = MW == 1 ? 0 : (int)(threadIdx.x >> 5) % MW;
  const int g = lane >> 2, t = lane & 3;
  LineGeom lg;
  lg.R = PENCIL ? p.Rp : p.R[axis];
  lg.PR = (long long)P * lg.R;
  lg.nlines = PENCIL ? p.Rp : p.nlines;
  Own<P, RIGHT> own[NT];
  long long base0[NT];
#pragma unroll
  for (int j = 0; j < NT; j++) {
    const long long nj = n0 + 8 * j;
    base0[j] = RIGHT ? nj * P : lg.base(nj);
    own[j].base = RIGHT ? (nj + g) * P : base0[j] + 2 * t;
    own[j].R = lg.R;
    own[j].g = g;
    own[j].t = t;
    own[j].r0 = h * TN * 8;
  }
  const double* __restrict__ g0 = PENCIL ? p.g0_p : p.g0[axis];
  const double* __restrict__ eta_a = PENCIL ? p.eta_p : p.eta;
  const double* __restrict__ deta_a = PENCIL ? p.deta_p : p.deta;
  const double* __restrict__ etap = XF(p, 1) ? nullptr : eta_a;
#ifdef SB200_TRACE
  long long* tr = p.trace ? p.trace + ((long long)axis * (p.nlines / (8 * NT)) + n0 / (8 * NT)) * 8 : nullptr;
  if (lane == 0 && p.trace) { unsigned smid; asm("mov.u32 %0, %%smid;" : "=r"(smid)); tr[6] = smid; tr[7] = threadIdx.x >> 5; }
#endif
  STAMP(0);
  FluxBuf f0, f1;
  if (DEEP) flux_load<P, RIGHT, TN>(f0, own[0], 0, etap, deta_a, g0);
#pragma unroll
  for (int j = 0; j < NT; j++) {
    prefetch_block<P, RIGHT, MW>(eta_a, base0[j], lg.R, lane, h);
    prefetch_block<P, RIGHT, MW>(deta_a, base0[j], lg.R, lane, h);
    prefetch_block<P, RIGHT, MW>(g0, base0[j], lg.R, lane, h);
    if (RIGHT && !PENCIL) {
      // last axis: the partial sums its epilogue adds (4 dependent batches of loads) are pulled into L2 now, a whole chain ahead
      for (int k = 0; k < p.d - 1; k++) prefetch_block<P, true, MW>(p.part[k], base0[j], 1, lane, h);
    }
  }
  cp_async_wait<0>();
  item_sync<MW>();  // (MW == 2: the other warp's half of the block has landed too)
  STAMP(1);

  double a[NT][TN][2], b[NT][TN][2];
  eo_gemm_nt<P, NT, RIGHT, TN>(Ae, Bo, Xw, a, b, g, t, h * TN);
  __syncwarp();
  STAMP(2);
#pragma unroll
  for (int j = 0; j < NT; j++) {
    double* Xj = Xw + j * BE;
    if (MW > 1) {
      // the first batch has been in flight since before GEMM1; registers hold one batch only, so the next is loaded after it is applied
      item_sync<MW>();  // the other warp's GEMM1 has read the rows overwritten below
#pragma unroll
      for (int ib = 0; ib < TN; ib += 2) {
        if (ib > 0) flux_load<P, RIGHT, TN>(f0, own[j], ib, etap, deta_a, g0);
        flux_apply<P, RIGHT, TN>(f0, own[j], ib, Xj, a[j], b[j]);
      }
    } else if (DEEP) {
      // software pipeline: batch k+1 is in flight while batch k is applied
      if (j > 0) flux_load<P, RIGHT, TN>(f0, own[j], 0, etap, deta_a, g0);
#pragma unroll
      for (int ib = 0; ib < TN; ib += 4) {  // (tiles ib, ib+1 always exist; ib+2, ib+3 only when TN % 4 == 0 or ib + 4 <= TN)
        if (ib + 2 < TN) flux_load<P, RIGHT, TN>(f1, own[j], ib + 2, etap, deta_a, g0);
        flux_apply<P, RIGHT, TN>(f0, own[j], ib, Xj, a[j], b[j]);
        if (ib + 4 < TN) flux_load<P, RIGHT, TN>(f0, own[j], ib + 4, etap, deta_a, g0);
        if (ib + 2 < TN) flux_apply<P, RIGHT, TN>(f1, own[j], ib + 2, Xj, a[j], b[j]);
      }
    } else {
#pragma unroll
      for (int ib = 0; ib < TN; ib += 2) {
        flux_load<P, RIGHT, TN>(f0, own[j], ib, etap, deta_a, g0);
        flux_apply<P, RIGHT, TN>(f0, own[j], ib, Xj, a[j], b[j]);
      }
    }
  }
  item_sync<MW>();  // (MW == 2: GEMM2 reads the rows the other warp has just written)
  STAMP(3);
  refill(0);
  eo_gemm_nt<P, NT, RIGHT, TN>(Ae, Bo, Xw, a, b, g, t, h * TN);
  refill(1);
  item_sync<MW>();  // block free again (the caller refills it while the epilogue drains)
  refill(2);
  STAMP(4);

  if (XF(p, 2)) {
    // experiment: no epilogue traffic (keep one dependent store so the GEMM is not dead code)
    if (a[0][0][0] + b[0][0][0] == 12345.678) p.V[0] = 1.0;
  } else if (PENCIL && NT == 1 && p.bulk) {
    // axis 0 of the slab partition: the item's P x 8 result block is staged in shared memory ([row][8 lines], 64 bytes per row) and
    // leaves as ONE TMA tensor store per destination rank (box = 8 lines x nloc planes of that rank's part[0] field): the rows
    // cross NVLink while this warp goes on with its next item
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // the previous item's rows have been read out of the staging block
    __syncwarp();
#pragma unroll
    for (int i = 0; i < E::MT; i++) {
      const int mt = i * 8 + g, mb = P - 1 - mt;
      st2(stage + mt * 8 + 2 * t, a[0][i][0] + b[0][i][0], a[0][i][1] + b[0][i][1]);
      st2(stage + mb * 8 + 2 * t, b[0][i][0] - a[0][i][0], b[0][i][1] - a[0][i][1]);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes visible to the TMA engine
    __syncwarp();
    if (lane < p.nranks) {
      const int nloc = 1 << p.lognloc;
      const int col = (int)((long long)p.rank * p.Rp + n0);  // first line of the block inside a plane
      tma_store_2d(&maps->m[lane], col, 0, stage + (lane << p.lognloc) * 8);
    }
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  } else if (PENCIL) {
    // axis 0 of the slab partition: rows of D f go to the part[0] array of the rank that owns the plane
    const int nloc = 1 << p.lognloc;
#pragma unroll
    for (int j = 0; j < NT; j++) {
      const long long col = (long long)p.rank * p.Rp + n0 + 8 * j + 2 * t;  // line index inside a plane
#pragma unroll
      for (int i = 0; i < E::MT; i++) {
        const int mt = i * 8 + g, mb = P - 1 - mt;
        const int qt = XF(p, 16) ? p.rank : mt >> p.lognloc, qb = XF(p, 16) ? p.rank : mb >> p.lognloc;
        st2(p.part0peer[qt] + (long long)(mt - qt * nloc) * p.R0 + col, a[j][i][0] + b[j][i][0], a[j][i][1] + b[j][i][1]);
        st2(p.part0peer[qb] + (long long)(mb - qb * nloc) * p.R0 + col, b[j][i][0] - a[j][i][0], b[j][i][1] - a[j][i][1]);
      }
    }
  } else if (!RIGHT) {
    // non-last axis: partial_k = D f
    double* __restrict__ part = p.part[axis];
#pragma unroll
    for (int j = 0; j < NT; j++) {
#pragma unroll
      for (int i = 0; i < TN; i++) {
        st2(part + own[j].top(i), a[j][i][0] + b[j][i][0], a[j][i][1] + b[j][i][1]);
        st2(part + own[j].bot(i), b[j][i][0] - a[j][i][0], b[j][i][1] - a[j][i][1]);
      }
    }
  } else {
    // last axis: phase A (all partials) must be complete and visible, then
    // V = crop(((0 - p_0) - p_1 ...) - D f)
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (WAITDONE) {
      if (lane == 0) {
        const long long t0 = clock64();
        while (*reinterpret_cast<volatile unsigned*>(p.sync + 6) < p.nlocal_items) {
          if (clock64() - t0 > SB200_SPIN_LIMIT) {
            symm_record_timeout(p.sf.f[p.rank]);
            break;
          }
        }
        __threadfence();
      }
      __syncwarp();
    }
    if (WAITDONE && !XF(p, 8)) {
      if (lane == 0) tl_stamp(p, 6);
      if (lane < p.nranks) spin_until(p.sf.f[p.rank] + SYMM_DONE + lane, p.epoch, p.sf.f[p.rank]);
      __syncwarp();
      if (lane == 0) tl_stamp(p, 7);
    }
#pragma unroll
    for (int j = 0; j < NT; j++) {
      long long n = n0 + 8 * j + g, gid = 0, mul = 1;
      bool vint = true;
      for (int q = p.d - 2; q >= 0; q--) {
        int iq;
        if (q == 0) {
          iq = (int)n + p.sg.i0;  // slowest digit: whatever remains (+ slab offset)
        } else {
          iq = (int)(n % P);
          n /= P;
        }
        const int ext = q == 0 ? p.sg.n0g : P;
        vint = vint && iq > 0 && iq < ext - 1;
        gid += (long long)(iq - 1) * mul;
        mul *= P - 2;
      }
      const long long vrow = gid * (P - 2) - p.sg.goff - 1;  // V index of row m is vrow + m
#pragma unroll
      for (int ib = 0; ib < TN; ib += 4) {  // (a split item at P = 128, TN = 4: one batch of loads per warp)
        double2 ot[4], ob[4];
#pragma unroll
        for (int ii = 0; ii < 4; ii++) ot[ii] = ob[ii] = make_double2(0.0, 0.0);
        if (p.d == 3) {
          // common case: both partials of the batch in flight at once
          double2 lt[2][4], lb[2][4];
#pragma unroll
          for (int k = 0; k < 2; k++) {
            const double* __restrict__ pk = p.part[k];
#pragma unroll
            for (int ii = 0; ii < 4; ii++) {
              if (ib + ii >= TN) continue;  // (TN % 4 != 0: the last batch is short)
              lt[k][ii] = __ldcg(reinterpret_cast<const double2*>(pk + own[j].top(ib + ii)));
              lb[k][ii] = __ldcg(reinterpret_cast<const double2*>(pk + own[j].bot(ib + ii)));
            }
          }
#pragma unroll
          for (int k = 0; k < 2; k++) {
#pragma unroll
            for (int ii = 0; ii < 4; ii++) {
              if (ib + ii >= TN) continue;
              ot[ii].x -= lt[k][ii].x;
              ot[ii].y -= lt[k][ii].y;
              ob[ii].x -= lb[k][ii].x;
              ob[ii].y -= lb[k][ii].y;
            }
          }
        } else {
          for (int k = 0; k < p.d - 1; k++) {
            const double* __restrict__ pk = p.part[k];
            double2 lt[4], lb[4];
#pragma unroll
            for (int ii = 0; ii < 4; ii++) {
              if (ib + ii >= TN) continue;
              lt[ii] = __ldcg(reinterpret_cast<const double2*>(pk + own[j].top(ib + ii)));
              lb[ii] = __ldcg(reinterpret_cast<const double2*>(pk + own[j].bot(ib + ii)));
            }
#pragma unroll
            for (int ii = 0; ii < 4; ii++) {
              if (ib + ii >= TN) continue;
              ot[ii].x -= lt[ii].x;
              ot[ii].y -= lt[ii].y;
              ob[ii].x -= lb[ii].x;
              ob[ii].y -= lb[ii].y;
            }
          }
        }
        if (vint) {
#pragma unroll
          for (int ii = 0; ii < 4; ii++) {
            const int i = ib + ii;
            if (i >= TN) continue;
            const double yt0 = a[j][i][0] + b[j][i][0], yt1 = a[j][i][1] + b[j][i][1];
            const double yb0 = b[j][i][1] - a[j][i][1], yb1 = b[j][i][0] - a[j][i][0];
            const int mt = own[j].r0 + i * 8 + 2 * t, mb = P - 2 - own[j].r0 - i * 8 - 2 * t;  // first row of each pair
            if (mt > 0) p.V[vrow + mt] = ot[ii].x - yt0;
            p.V[vrow + mt + 1] = ot[ii].y - yt1;
            p.V[vrow + mb] = ob[ii].x - yb0;
            if (mb + 1 < P - 1) p.V[vrow + mb + 1] = ob[ii].y - yb1;
          }
        }
      }
    }
  }
  STAMP(5);
}

// Forward all-to-all of the slab partition, folded into the head of phase A: this CTA pads its share of
// the local input vector (zero Dirichlet rows, elliptic.C:305-308) and pushes plane (i0 + ml), lines
// [q*Rp, (q+1)*Rp) into rank q's pencil with 16-byte stores that are contiguous along the last axis.
template <int P>
__device__ __forceinline__ void stage_push_share(const PersistParams& p, int warp, int nwarps) {
  constexpr int LB = 4;        // lines in flight per warp: all their loads are issued before the first store
  constexpr int IT = (P + 63) / 64;  // 16-byte chunks per lane and line
  const int d = p.d, lane = threadIdx.x & 31;
  const unsigned nloc = 1u << p.lognloc;
  const unsigned lpp = (unsigned)(p.R0 / P), nl = nloc * lpp;  // lines per plane, local lines
  const unsigned per = (nl + gridDim.x - 1) / gridDim.x;
  const unsigned l0 = blockIdx.x * per, l1 = l0 + per < nl ? l0 + per : nl;
  const unsigned Rp = (unsigned)p.Rp;
  const double* __restrict__ U = p.U;
  for (unsigned base = l0 + warp * LB; base < l1; base += nwarps * LB) {
    double v[LB][IT][2];
    double* dst[LB][IT];
#pragma unroll
    for (int b = 0; b < LB; b++) {
      const unsigned line = base + b;
      const bool live = line < l1;
      const unsigned ml = line / lpp, lin = line - ml * lpp;
      unsigned rem = lin;
      long long gid = 0, ist = P - 2;
      bool inter = live;
      for (int j = d - 2; j >= 1; j--) {
        const int ij = (int)(rem % P);
        rem /= P;
        inter = inter && ij >= 1 && ij <= P - 2;
        gid += (long long)(ij - 1) * ist;
        ist *= (P - 2);
      }
      const int i0g = (int)ml + p.sg.i0;
      inter = inter && i0g >= 1 && i0g <= p.sg.n0g - 2;
      gid += (long long)(i0g - 1) * ist - p.sg.goff;  // ist == istride[0] here
#pragma unroll
      for (int it = 0; it < IT; it++) {
        const int k = 2 * lane + 64 * it;
        v[b][it][0] = (inter && k >= 1 && k <= P - 2) ? U[gid + k - 1] : 0.0;
        v[b][it][1] = (inter && k + 1 <= P - 2) ? U[gid + k] : 0.0;
        const unsigned n = lin * P + k, q = n / Rp;
        dst[b][it] = (live && k < P) ? p.wppeer[q] + (long long)i0g * Rp + (n - q * Rp) : nullptr;
      }
    }
#pragma unroll
    for (int b = 0; b < LB; b++)
#pragma unroll
      for (int it = 0; it < IT; it++)
        if (dst[b][it]) st2(dst[b][it], v[b][it][0], v[b][it][1]);
  }
}

// The forward all-to-all as its own small kernel (no shared memory, so its CTAs share the SMs with phase A,
// which is launched as a programmatic dependent and runs the local-axis items while the planes cross
// NVLink).  The last block to finish raises READY on every rank.
// Blocks are small (128 threads, <= 80 registers) because phase A's CTA already takes ~53K of the SM's 64K
// registers: only then do the two kernels really share an SM.
template <int P>
__global__ void __launch_bounds__(128, 6) stage_kernel(PersistParams p) {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  stage_push_share<P>(p, threadIdx.x >> 5, blockDim.x >> 5);
  if (threadIdx.x == 0) tl_stamp(p, 1);
  __syncthreads();  // the block's pushes happen-before thread 0's fence
  if (threadIdx.x == 0) {
    __threadfence_system();
    tl_stamp(p, 2);
    if (atomicAdd(p.sync + 3, 1u) == gridDim.x - 1) {
      p.sync[3] = 0;
      __threadfence_system();
      for (int q = 0; q < p.nranks; q++) st_relaxed_sys(p.sf.f[q] + SYMM_READY + p.rank, p.epoch);
    }
  }
}

// Register budget: one CTA per SM.  The slab kernel keeps ~9.7K registers of the SM free so that
// the blocks of the stage kernel (128 threads x 76 registers) can share the SM with it (PDL overlap).
constexpr int persist_maxreg(int nwarps, bool slab) {
  return nwarps > 8 ? (65536 / (nwarps * 32)) / 8 * 8 : (slab ? 216 : 255);
}

// MW: warps per item (1, or 2 on one GPU: a pair of warps splits the item's pair tiles, see run_item).
// SLAB: one launch for every axis of a slab rank - the local axes, the axis-0 pencil items, then the last axis (LASTPHASE is false).
template <int P, int NWARPS, int NT, int MW, bool LASTPHASE, bool SLAB>
__global__ void __maxnreg__(persist_maxreg(NWARPS, SLAB)) persist_kernel(PersistParams p, const __grid_constant__ SlabMaps maps) {
  using E = EO<P>;
  static_assert(!(SLAB && LASTPHASE), "slab: the last axis runs in the same launch");
  static_assert(MW == 1 || (!SLAB && NWARPS % MW == 0 && NWARPS / MW <= 15), "pairs: single GPU, one named barrier each");
  constexpr int NSLOT = NWARPS / MW;  // items in flight per CTA
  extern __shared__ __align__(128) double sm[];
  __shared__ unsigned next_ticket[NSLOT];  // MW == 2: the pair's next ticket, taken by its first warp
  double* Ae = sm;
  double* Bo = sm + E::H * E::LDM;
  constexpr int BEMAX = E::BLOCK_ELEMS_RIGHT > E::BLOCK_ELEMS_LEFT ? E::BLOCK_ELEMS_RIGHT : E::BLOCK_ELEMS_LEFT;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int slot = warp / MW, h = warp % MW;
  double* Xw = sm + E::MAT_ELEMS + slot * (NT * BEMAX);
  // slab: a staging block per warp for the pencil items' TMA stores (never touched by the loaders)
  double* stage = SLAB ? sm + E::MAT_ELEMS + NWARPS * (NT * BEMAX) + warp * (P * 8) : nullptr;
  unsigned* sync = p.sync + (LASTPHASE ? 4 : 0);  // [0] ticket, [1] exited warps

  const unsigned items_per_axis = (unsigned)(p.nlines / (8 * NT));
  // slab: the local axes come first; the axis-0 pencil items follow once every rank's planes have arrived (tickets
  // [nlocal, nlocal + items0)), the last-axis items come last
  const unsigned items0 = SLAB ? (unsigned)(p.Rp / (8 * NT)) : 0u;
  const unsigned nlocal = LASTPHASE ? items_per_axis : items_per_axis * (p.d - 1 - p.first_axis);
  const unsigned total = nlocal + items0 + (SLAB ? items_per_axis : 0u);
  if (!LASTPHASE) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  load_matrices<P>(sm, p.Ae, p.Bo);
  if (SLAB && threadIdx.x == 0) tl_stamp(p, 0);

  // First ticket: static, strided over the CTAs first (warp w of CTA c takes w * gridDim.x + c), so that with fewer
  // items than warps (a slab rank at 4 or 8 GPUs) every SM sub-partition gets at most one busy warp instead of the
  // first CTAs taking everything.  Later tickets come from the global counter, which starts behind the static ones.
  const unsigned nstatic = gridDim.x * NSLOT;
  auto grab = [&]() -> unsigned {
    unsigned tk = 0;
    if (lane == 0) tk = atomicAdd(sync, 1u) + nstatic;
    return __shfl_sync(0xffffffffu, tk, 0);
  };
  const unsigned first_ticket = slot * gridDim.x + blockIdx.x;
  bool peers_ready = false;
  auto issue_load = [&](unsigned tk) {
    if (tk >= total) return;
    if (SLAB && tk >= nlocal + items0) {
      load_item<P, NT, true>(Xw, p.U, p.d, p.d - 1, (long long)(tk - nlocal - items0) * (8 * NT), lane, p.sg);
      return;
    }
    if (SLAB && tk >= nlocal) {
      if (!peers_ready && !XF(p, 4)) {
        // every rank must have pushed its planes of the padded input into this rank's pencil
        if (lane < p.nranks) spin_until(p.sf.f[p.rank] + SYMM_READY + lane, p.epoch, p.sf.f[p.rank]);
        __syncwarp();
        if (lane == 0) tl_stamp(p, 3);
        peers_ready = true;
      }
      LineGeom lg;
      lg.R = p.Rp;
      lg.PR = (long long)P * p.Rp;
      lg.nlines = p.Rp;
#pragma unroll
      for (int j = 0; j < NT; j++)
        load_block<P, false>(Xw + j * E::BLOCK_ELEMS_LEFT, p.Wp, lg, (long long)(tk - nlocal) * (8 * NT) + 8 * j, lane);
      return;
    }
    const unsigned tl = tk;
    const int arel = LASTPHASE ? 0 : tl / items_per_axis;
    const int axis = LASTPHASE ? p.d - 1 : p.first_axis + arel;
    const long long n0 = (long long)(tl - arel * items_per_axis) * (8 * NT);
    load_item<P, NT, LASTPHASE, MW>(Xw, p.U, p.d, axis, n0, lane, p.sg, h);
  };

  constexpr bool DEEP = MW > 1 || (NWARPS * NT <= 8);  // 255 registers available, or a quarter of the item's accumulators per warp
  // De-phase the warps of each SM sub-partition (warp w runs on SMSP w % 4): identical items started
  // together stay in lockstep, which serialises the tensor phases against the memory phases.
  unsigned tk = 0;
  if (SLAB) {
    // a first ticket may be a pencil item that waits for the peers: never hold the CTA barrier behind it
    cp_async_wait<0>();
    __syncthreads();
    tk = first_ticket;
    issue_load(tk);
  } else {
    tk = first_ticket;
    issue_load(tk);
    cp_async_wait<0>();
    __syncthreads();  // matrices visible to all warps (the only CTA-wide barrier)
  }
  if (p.stagger > 0) {
    const long long until = clock64() + (long long)(warp / 4) * p.stagger;
    while (clock64() < until) {
    }
  }

  unsigned pencil_done = 0;  // pencil items this warp has finished and not yet reported
  auto report_pencils = [&]() {
    // all pushes of this warp are out; the rank whose last pencil item this was raises DONE everywhere
    if (p.bulk) {
      asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // this lane's tensor stores have completed (writes performed)
      asm volatile("fence.proxy.async.global;" ::: "memory");
      __syncwarp();
    }
    __threadfence_system();
    if (lane == 0) {
      const unsigned before = atomicAdd(sync + 2, pencil_done);
      if (before + pencil_done == items0) {
        tl_stamp(p, 4);
        sync[2] = 0;
        __threadfence_system();
        for (int q = 0; q < p.nranks; q++) st_relaxed_sys(p.sf.f[q] + SYMM_DONE + p.rank, p.epoch);
      }
    }
    pencil_done = 0;
  };
  unsigned nxt = 0;
  while (tk < total) {
    if (SLAB && tk >= nlocal + items0) {
      if (pencil_done) report_pencils();  // before this warp may block on the other ranks' DONE
      run_item<P, NT, true, DEEP, 1, false, true>(p, p.d - 1, (long long)(tk - nlocal - items0) * (8 * NT), Ae, Bo, Xw, lane);
    } else if (SLAB && tk >= nlocal) {
      run_item<P, NT, false, DEEP, 1, true>(p, 0, (long long)(tk - nlocal) * (8 * NT), Ae, Bo, Xw, lane, &maps, stage);
      pencil_done++;
    } else {
      const unsigned tl = tk;
      const int arel = LASTPHASE ? 0 : tl / items_per_axis;
      const int axis = LASTPHASE ? p.d - 1 : p.first_axis + arel;
      const long long n0 = (long long)(tl - arel * items_per_axis) * (8 * NT);
      if (SLAB) {
        run_item<P, NT, false, DEEP, 1>(p, axis, n0, Ae, Bo, Xw, lane);
      } else {
        unsigned claimed = 0;
        auto early = [&](int at) {
          if (MW == 1) {
            if (at == 2) {
              nxt = grab();
              issue_load(nxt);
            }
          } else if (at == 0) {
            if (h == 0 && lane == 0) claimed = atomicAdd(sync, 1u) + nstatic;  // one ticket per pair; its latency hides behind GEMM2
          } else if (at == 1) {
            if (h == 0 && lane == 0) next_ticket[slot] = claimed;  // published by the pair barrier that follows
          } else {
            nxt = next_ticket[slot];
            issue_load(nxt);  // both warps load their half of the block
          }
        };
        run_item<P, NT, LASTPHASE, DEEP, MW>(p, axis, n0, Ae, Bo, Xw, lane, nullptr, nullptr, early);
      }
      if (SLAB) {
        __threadfence();  // this item's partial rows are visible device-wide before it checks in
        __syncwarp();
        if (lane == 0) atomicAdd(sync + 6, 1u);
      }
    }
    if (SLAB) {
      tk = grab();
      issue_load(tk);  // run_item waits for it at its top
    } else {
      tk = nxt;  // grabbed and loading since the end of GEMM2
    }
  }
  cp_async_wait<0>();
  if (SLAB && pencil_done) report_pencils();
  // the last warp to leave re-arms the counters for the next launch
  if (lane == 0) {
    const unsigned gone = atomicAdd(sync + 1, 1u);
    if (gone == gridDim.x * NWARPS - 1) {
      sync[0] = 0;
      sync[1] = 0;
      if (SLAB) {
        sync[6] = 0;
        tl_stamp(p, 8);
      }
    }
  }
}

// Test hook SB200_MAX_CTAS: caps the grids, so that several slab ranks emulated on ONE device are all resident at the same time.
long long cap_ctas(long long grid) {
  const char* mc = getenv("SB200_MAX_CTAS");
  const int lim = mc ? atoi(mc) : 0;
  return lim > 0 && grid > lim ? lim : grid;
}

template <int P, int NWARPS, int NT, int MW, bool LASTPHASE, bool SLAB>
int launch_phase(const PersistParams& p, size_t smem, int sms, cudaStream_t s) {
  auto kern = persist_kernel<P, NWARPS, NT, MW, LASTPHASE, SLAB>;
  static bool attr[64] = {};  // the opt-in above 48 KB of dynamic shared memory is per device
  int cur = 0;
  cudaGetDevice(&cur);
  if (!attr[cur & 63]) {
    SB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr[cur & 63] = true;
  }
  long long items = p.nlines / (8 * NT) * (LASTPHASE ? 1 : p.d - 1 - p.first_axis);
  if (SLAB) items += p.Rp / (8 * NT) + p.nlines / (8 * NT);
  if (items <= 0) return 0;
  // one persistent CTA per SM; with fewer items than warps spread them over all SMs (a warp alone on its
  // SM sub-partition issues DMMAs ~1.5x faster than two sharing it)
  long long grid = cap_ctas(items < sms ? items : sms);
  if (grid < 1) grid = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(NWARPS * 32);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  // phase B may start while phase A drains; the slab kernel may start while the stage kernel pushes
  cfg.numAttrs = (LASTPHASE || SLAB) ? 1 : 0;
  static const SlabMaps no_maps = {};
  SB_CUDA(cudaLaunchKernelEx(&cfg, kern, p, (SLAB && p.maps) ? *p.maps : no_maps));
  count_launch();
  return 0;
}

template <int P, int NWARPS, int NT, int MW = 1>
int run_cfg(PersistParams& p, cudaStream_t s) {
  using E = EO<P>;
  constexpr int BEMAX = E::BLOCK_ELEMS_RIGHT > E::BLOCK_ELEMS_LEFT ? E::BLOCK_ELEMS_RIGHT : E::BLOCK_ELEMS_LEFT;
  const size_t smem = (size_t)(E::MAT_ELEMS + NWARPS / MW * NT * BEMAX) * sizeof(double);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  // start stagger per group of 4 warps (clk): split items 3000 (0 / 3000 / 6000: 0.107 / 0.089 / 0.093 ms at 128^3, profiles/r03_notes.md),
  // whole items 6000 (profiles/r02_notes.md)
  p.stagger = MW > 1 ? 3000 : 6000;
  if constexpr (MW > 1) {
    SB_CHECK(p.nranks == 1, SB200_ERR_SUP, "persistent path: split items are a single-GPU configuration");
  } else if (p.nranks > 1) {
    const size_t smem_slab = smem + (size_t)NWARPS * P * 8 * sizeof(double);  // + the pencil items' staging blocks
    if (!XF(p, 32)) {
      const int blocks = (int)cap_ctas(sms);
      {
        // same shared-memory carve-out as the chain kernel that shares the SMs with it: an SM whose carve-out has to change
        // first drains, which delayed the chain kernel's CTAs behind the stage blocks (CTA starts spread over 12 us at 2 GPUs)
        static bool carve[64] = {};
        if (!carve[dev & 63]) {
          cudaFuncSetAttribute(stage_kernel<P>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
          carve[dev & 63] = true;
        }
      }
      stage_kernel<P><<<blocks, 128, 0, s>>>(p);
      count_launch();
      SB_CUDA(cudaGetLastError());
    }
    p.nlocal_items = (unsigned)(p.nlines / (8 * NT) * (p.d - 1 - p.first_axis));
    if (NT != 1) p.bulk = 0;
    return launch_phase<P, NWARPS, NT, 1, false, true>(p, smem_slab, sms, s);
  }
  SB_TRY((launch_phase<P, NWARPS, NT, MW, false, false>(p, smem, sms, s)));
  SB_TRY((launch_phase<P, NWARPS, NT, MW, true, false>(p, smem, sms, s)));
  return 0;
}

}  // namespace

bool elliptic_persist_supported(const EllipticCtx& e) {
  const int d = e.gd.d;
  if (d < 2 || e.arena.nranks > 1) return false;
  const int P = e.gd.dim[0];
  for (int j = 1; j < d; j++)
    if (e.gd.dim[j] != P) return false;
  return P % 16 == 0 && P >= 32 && P <= 160 && (e.gd.m / P) % 16 == 0;
}

int persist_run(int P, PersistParams& p, cudaStream_t s) {
#ifdef SB200_ABLATE
  const char* xf = getenv("SB200_XFLAGS");
  p.xflags = xf ? atoi(xf) : 0;
  const char* tl = getenv("SB200_TL_EPOCH");
  p.tl_epoch = tl ? (unsigned long long)atoll(tl) : 0;
#else
  p.xflags = 0;
#endif
  SB_CHECK(p.nlines % 16 == 0, SB200_ERR_SUP, "persistent path: line count must be a multiple of 16");
  switch (P) {
    case 32: return run_cfg<32, 16, 1>(p, s);
    case 64: return run_cfg<64, 16, 1>(p, s);
    // the extents between the powers of two: single-GPU instantiations of the same kernel (no extent cliff for P % 16 == 0 up to 160)
    case 48: SB_CHECK(p.nranks == 1, SB200_ERR_SUP, "persistent path: this extent is a single-GPU instantiation"); return run_cfg<48, 16, 1>(p, s);
    case 80: SB_CHECK(p.nranks == 1, SB200_ERR_SUP, "persistent path: this extent is a single-GPU instantiation"); return run_cfg<80, 12, 1>(p, s);
    case 96: SB_CHECK(p.nranks == 1, SB200_ERR_SUP, "persistent path: this extent is a single-GPU instantiation"); return run_cfg<96, 12, 1>(p, s);
    case 112: SB_CHECK(p.nranks == 1, SB200_ERR_SUP, "persistent path: this extent is a single-GPU instantiation"); return run_cfg<112, 12, 1>(p, s);
    case 144: SB_CHECK(p.nranks == 1, SB200_ERR_SUP, "persistent path: this extent is a single-GPU instantiation"); return run_cfg<144, 8, 1>(p, s);
    case 160: SB_CHECK(p.nranks == 1, SB200_ERR_SUP, "persistent path: this extent is a single-GPU instantiation"); return run_cfg<160, 8, 1>(p, s);
    case 128:
      // one GPU: 8 pairs of warps x 128 registers, each pair splitting one item (0.089 ms against 0.099 ms for 12 whole-item warps x 168
      // registers on a B200 at 1000 W, profiles/r03_notes.md; split items at P = 64 / 96 measured slower, at 32 equal); a slab partition
      // keeps 8 whole-item warps x 255 (its staging blocks need the shared memory of further warps' blocks)
      if (p.nranks > 1) return run_cfg<128, 8, 1>(p, s);
      return run_cfg<128, 16, 1, 2>(p, s);
  }
  set_last_error("persistent path: unsupported extent");
  return SB200_ERR_SUP;
}

int elliptic_matmult_persist(EllipticCtx& e, const double* U, double* V, cudaStream_t s) {
  const int P = e.gd.dim[0], d = e.gd.d;
  if (!e.sync) {
    SB_CUDA(cudaMalloc((void**)&e.sync, 512));
    SB_CUDA(cudaMemsetAsync(e.sync, 0, 512, s));
  }
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
  p.sg.i0 = 0;
  p.sg.n0g = P;
  p.sg.goff = 0;
  p.first_axis = 0;
  p.nranks = 1;
  p.rank = 0;
  p.trace = e.trace;
  return persist_run(P, p, s);
}

}  // namespace sb200
