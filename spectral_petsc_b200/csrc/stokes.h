// Internal: device-side context for the stokes.C shells (replaces StokesCtx, stokes.C:40-65).
#pragma once
#include <cuda_runtime.h>

#include <vector>

#include "deriv.h"
#include "elliptic.h"  // GridDesc, DiffMatrix

extern "C" typedef int (*sb200_velocity_solve_fn)(void* ctx, const double* d_rhs, double* d_sol, void* stream);

namespace sb200 {

struct StokesCtx {
  GridDesc gd;
  long long gp = 0, gv = 0, g = 0, dvn = 0;  // DOF counts printed at stokes.C:891
  double* workV[2 + 3 + 1] = {};  // xL, yL, V[d], one more term buffer   (c->workV, stokes.C:271)
  double* workP[3] = {};      // pL, scratch, accumulator (c->workP)
  double* strain[3] = {};     // c->strain, each m*d
  double* eta = nullptr;
  double* deta = nullptr;
  double* dirichlet = nullptr;  // dv values: boundary nodes in walk order x d components
  double* force = nullptr;      // c->force (g)
  double* vG0 = nullptr;        // c->vG0 / vG1 (used by the Schur shell)
  double* vG1 = nullptr;
  double* minmax = nullptr;     // device [min eta, max eta] of the last residual evaluation
  double* w0[3] = {};           // end-point extrapolation weights per axis (StokesPressureReduceOrder)
  double* w1[3] = {};
  int rheology = 0;             // 0 linear, 1 power law (stokes.C:481-492)
  double hardness = 1.0, exponent = 1.0, regularization = 1.0, gamma0 = 1.0;
  DiffMatrix* Dax[3] = {};
  std::vector<DiffMatrix*> owned;
  std::vector<double*> owned_w;
  // slab partition along axis 0 (nranks == 1: single GPU); the exchangeable arrays live in the arena
  SymmArena arena;
  int gdim[3] = {};
  unsigned* sync = nullptr;  // counters of the even-odd derivative kernel
  double* Xp = nullptr;   // pencil operand / result buffers of the axis-0 derivative (m*d doubles each)
  double* Yp = nullptr;
  // slab: the local-axis derivative batch runs here, beside the axis-0 pencil chain on the caller's stream; single GPU: the folded pressure
  cudaStream_t aux_stream = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_pjoin = nullptr;
  bool pressure_pending = false;  // the folded pressure is being prepared on the side stream (join_pressure before its consumer)
  int fold_pressure_begin(const double* xG, cudaStream_t s);
  int join_pressure(cudaStream_t s);
  double* red = nullptr;  // [nranks][2][lines per plane]: partial end-point sums of the axis-0 extrapolation pass

  static int create(int d, const int* dim, int rank, int nranks, StokesCtx** out);
  int init(int d, const int* dim, int rank, int nranks);
  ~StokesCtx();
  int deriv_common(struct DerivParams& p, int axis, cudaStream_t s);
  DerivParams job_v(int axis, const double* x, double* y, const double* yin, int mode) const;
  DerivParams job_p(int axis, const double* x, int xs, int xoff, double* y, int ys, int yoff, const double* yin, int mode) const;
  // true when the d derivatives can run as one even-odd launch (single GPU, equal extents in {16,32,64,128})
  bool batchable() const;
  // single GPU and every extent <= SB200_EO_MAX_P: pad / crop / AXPY chains run inside the derivative launches (deriv.h)
  bool fusable() const;
  EoLineMap line_map(int axis, int nc) const;
  int run_jobs(DerivParams* jobs, int d, cudaStream_t s);
  int crop_sum(int nc, int nterms, double* const* terms, double sign, double* dst, int dstride, int doff, cudaStream_t s);

  int deriv_v(int axis, const double* x, double* y, const double* yin, int mode, cudaStream_t s);
  int deriv_p(int axis, const double* x, int xs, int xoff, double* y, int ys, int yoff, const double* yin, int mode,
              cudaStream_t s);
  int pad_vel(const double* src, int sstride, int soff, bool with_dirichlet, double* local, cudaStream_t s);
  int pad_pres(const double* src, int sstride, int soff, double* local, cudaStream_t s);
  int crop(int nc, const double* local, double* dst, int dstride, int doff, bool add, const double* sub, cudaStream_t s);
  int viscous_tail(double* dst, int dstride, int doff, cudaStream_t s);
  // div_dst != nullptr: also write  sum_i D_i v_i  (the trace of the velocity gradient this shell computes anyway) into
  // div_dst[gid*div_stride + div_off] - what a following StokesMatMultPV on the same input would compute a second time
  int matmult_vv_into(const double* x, int xstride, int xoff, double* dst, int dstride, int doff, cudaStream_t s,
                      double* div_dst = nullptr, int div_stride = 0, int div_off = 0, const double* p_local = nullptr);
  int crop_trace(double* const* grads, double* dst, int dstride, int doff, cudaStream_t s);
  // Evaluation switch (sb200_stokes_set_trace_divergence; ON by default since round 2: measured and parity-tested at 128^3,
  // profiles/r02_notes.md; off = the reference's literal sequence of shells): StokesMatMult and StokesFunction take
  // their pressure rows from the trace of the velocity gradient of the viscous block instead of padding the same velocity and
  // differentiating its components again (stokes.C:509,746 call StokesDivergence on the input the gradient was just taken of).
  bool trace_divergence = true;
  // Evaluation switch (sb200_stokes_set_fold_pressure; ON by default since round 2): StokesMatMult and StokesFunction subtract the padded,
  // boundary-extrapolated pressure from the diagonal of the viscous flux (V = eta*eps - p I, the stress), so the one divergence
  // of the viscous tail also yields the pressure gradient and StokesMatMultVP's d derivative passes and its add-crop disappear.
  // Same operator; the sum -D_j V_jj + D_j p is rounded once instead of twice (differences ~1e-15 relative).
  bool fold_pressure = true;
  int divergence_into(const double* x, int xstride, int xoff, bool with_dirichlet, double* dst, int dstride, int doff,
                      cudaStream_t s);
  int pressure_reduce_order(double* pL, cudaStream_t s, int first_pass = 0);
  int pad_pres_reduced(const double* src, int sstride, int soff, double* pL, cudaStream_t s);
  int matmult_vp_into(const double* x, int xstride, int xoff, double* dst, int dstride, int doff, bool add,
                      const double* sub, cudaStream_t s);
  int matmult(const double* xG, double* yG, cudaStream_t s);
  int function(const double* xG, double* yG, cudaStream_t s);
  int get_diagonal_schur(double* y, cudaStream_t s);
  int matmult_schur(const double* x, double* y, sb200_velocity_solve_fn solve, void* solve_ctx, cudaStream_t s);
};

int axpy_launch(long long n, double a, const double* x, double* y, cudaStream_t s);

}  // namespace sb200
