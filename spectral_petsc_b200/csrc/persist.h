// Internal: parameters of the persistent chain kernels (elliptic_persist.cu), shared with the slab
// (multi-GPU) driver in elliptic_slab.cu.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include "elliptic.h"

namespace sb200 {

// Slab view of axis 0 for the multi-GPU partition: the local array holds planes [i0, i0+nloc) of a
// global grid whose axis 0 has extent n0g; goff = global id of the first locally stored interior node.
// Single GPU: i0 = 0, n0g = P, goff = 0.
struct SlabGeom {
  int i0, n0g;
  long long goff;
};

struct PersistParams {
  const double* Ae;
  const double* Bo;
  const double* U;     // global vector (g): the pad is applied by the block loader
  const double* eta;   // m
  const double* deta;  // m
  const double* g0[SB200_MAX_DIM];   // gradu[k]
  double* part[SB200_MAX_DIM];       // partial fields of the non-last axes
  double* V;                         // g: cropped result
  long long R[SB200_MAX_DIM];        // stride of axis k
  long long nlines;                  // m / P (same for every axis)
  int d;
  unsigned* sync;  // phase A: [0] ticket, [1] exited warps; phase B: [4], [5]
  SlabGeom sg;       // axis-0 slab view (single GPU: {0, P, 0})
  int first_axis;    // phase A runs axes first_axis..d-2 (0; 1 in slab mode where axis 0 is exchanged)
  // ---- slab mode (nranks > 1): axis 0 runs on "pencils" (all P planes of R0/nranks lines) --------
  int nranks, rank, lognloc;            // nloc = P / nranks = 1 << lognloc planes per rank
  const double* Wp;                     // this rank's pencil [P][Rp] of the padded input, pushed by all ranks
  double* wppeer[SB200_MAX_RANKS];      // Wp of every rank (forward all-to-all: planes are pushed at kernel start)
  double* part0peer[SB200_MAX_RANKS];   // part[0] (slab layout) of every rank: axis-0 results are pushed
  const double* eta_p;                  // pencil-layout copies [P][Rp] of eta / deta / gradu[0]
  const double* deta_p;
  const double* g0_p;
  long long R0, Rp;                     // lines per plane; lines per pencil (R0 / nranks)
  SymmFlags sf;
  unsigned long long epoch;             // READY / DONE flag value of this application
  int bulk;                             // slab: pencil results leave through TMA tensor stores (maps != nullptr) instead of per-thread stores
  const SlabMaps* maps;                 // host pointer (copied into the kernel's __grid_constant__ parameter at launch)
  unsigned nlocal_items;                // slab: local (non-pencil, non-last-axis) items whose partials the last axis reads
  unsigned long long tl_epoch;          // debug timeline (diagnostic builds): the application to stamp (SB200_TL_EPOCH)
  int stagger;       // start delay per warp group, in clocks
  int xflags;        // experiment switches (0 in production): 1 = no flux loads, 2 = no epilogue traffic
  long long* trace;  // optional (SB200_TRACE builds): per-item phase time stamps
};

// TMA descriptors of every rank's part[0] field viewed as [nloc planes][R0 lines] (fp64), box = 8 lines x nloc planes: the pencil
// epilogue stages an item's result rows in shared memory and ONE cp.async.bulk.tensor store per destination rank carries the rows
// that rank owns over NVLink - the issuing warp does not wait for the wire.  Passed to the kernel as a __grid_constant__ parameter.
struct alignas(64) SlabMaps {
  CUtensorMap m[SB200_MAX_RANKS];
};

// Single GPU: runs phase A (axes 0..d-2) and phase B (last axis).  Slab mode: one launch runs the local axes, the
// axis-0 pencil items and the last axis, extent P in {32, 64, 128}.
int persist_run(int P, PersistParams& p, cudaStream_t s);

}  // namespace sb200
