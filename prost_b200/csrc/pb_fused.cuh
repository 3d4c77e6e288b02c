// pb_fused.cuh -- fused PDHG passes.
//
// One PDHG iteration of the reference (backend_pdhg.cu:311-381) is >= 8 kernels over 9 state
// vectors.  Here it is two passes over 4 state vectors:
//
//   primal pass  x+ = prox_g( x - tau T (K^T y) )          K^T y gathered pointwise from y
//   dual pass    y+ = prox_f*( y + sigma S ((1+theta) K x+ - theta K x) )   K x+, K x gathered
//
// Each pass is prox_pass_kernel (pb_prox.cuh) with a Source that computes the prox argument on
// the fly from the block descriptors (pb_linop.cuh).  On residual iterations the same passes
// also accumulate the reference's residual sums (backend_pdhg.cu:73-120, 392-431):
//   dual residual   (primal pass): w^ = (x - x+)/(tau sqrt T) - sqrt T K^T y_prev ; diff = w^ + sqrt T K^T y
//   primal residual (dual pass)  : z^ = (y - y+)/(sigma sqrt S) + sqrt S ((1+th) Kx+ - th Kx) ; diff = z^ - sqrt S Kx+
// with K^T y_prev gathered from the previous dual iterate, which is still resident in the
// ping-pong buffer.  Reference quirks kept: K^T y is taken as 0 during iteration 0 (it is never
// computed from y0), K^T y_prev as 0 during iterations 0 and 1, and K x_prev as 0 during
// iteration 0 (Appendix B #1, #3 of SURVEY.md).
#pragma once

#include "pb_backend.cuh"
#include "pb_linop.cuh"
#include "pb_prox.cuh"
#include "pb_reduce.cuh"

namespace pb {

constexpr int kMaxFusedBlocks = 6;

struct SlabHalo;   // pb_comm.cuh

struct BlockList {
  int n = 0;
  BlockDesc b[kMaxFusedBlocks];
};

#ifdef __CUDACC__

// (K^T p)[e] for a global column index e
__device__ __forceinline__ float gather_col(const BlockList& bl, uint32_t e, const float* __restrict__ p) {
  float acc = 0.f;
  for (int k = 0; k < bl.n; ++k) {
    const BlockDesc& b = bl.b[k];
    if (e >= b.col && e - b.col < b.ncols) acc += block_col_dot(b, e - b.col, p + b.row);
  }
  return acc;
}

// (K u)[e] for a global row index e
__device__ __forceinline__ float gather_row(const BlockList& bl, uint32_t e, const float* __restrict__ u) {
  float acc = 0.f;
  for (int k = 0; k < bl.n; ++k) {
    const BlockDesc& b = bl.b[k];
    if (e >= b.row && e - b.row < b.nrows) acc += block_row_dot(b, e - b.row, u + b.col);
  }
  return acc;
}

template <int CAP, bool CHECK>
struct PrimalSource {
  const float* __restrict__ x;        // x^k
  const float* __restrict__ y;        // y^k
  const float* __restrict__ y_prev;   // y^{k-1} (CHECK only)
  ScaleRef T;
  const PdhgState* __restrict__ st;
  BlockList bl;
  int kty_zero, ktyprev_zero;
  double* __restrict__ partials;      // [gridDim.x][2], CHECK only

  struct Regs {
    float tau;
    float xo[CHECK ? CAP : 1], kty[CHECK ? CAP : 1], ktyp[CHECK ? CAP : 1];
    double acc0, acc1;
  };

  __device__ __forceinline__ float begin(Regs& r) const {
    r.tau = st->tau;
    r.acc0 = r.acc1 = 0.0;
    return r.tau;
  }
  __device__ __forceinline__ float load(Regs& r, uint32_t e, int i) const {
    const float xv = x[e];
    const float k = kty_zero ? 0.f : gather_col(bl, e, y);
    if (CHECK) {
      r.xo[i] = xv;
      r.kty[i] = k;
      r.ktyp[i] = ktyprev_zero ? 0.f : gather_col(bl, e, y_prev);
    }
    return primal_prox_arg(xv, r.tau, T.at(e), k);
  }
  __device__ __forceinline__ void post(Regs& r, uint32_t e, int i, float xn) const {
    if (CHECK) {
      const float sq = sqrtf(T.at(e));
      const float w_hat = (r.xo[i] - xn) / (r.tau * sq) - sq * r.ktyp[i];
      const float diff = w_hat + sq * r.kty[i];
      r.acc0 += static_cast<double>(diff * diff);
      r.acc1 += static_cast<double>(w_hat * w_hat);
    }
  }
  __device__ __forceinline__ void finish(Regs& r) const {
    if (CHECK) {
      block_sum2(r.acc0, r.acc1);
      if (threadIdx.x == 0) { partials[2 * blockIdx.x] = r.acc0; partials[2 * blockIdx.x + 1] = r.acc1; }
    }
  }
};

template <int CAP, bool CHECK>
struct DualSource {
  const float* __restrict__ y;        // y^k
  const float* __restrict__ x_new;    // x^{k+1}
  const float* __restrict__ x_old;    // x^k
  ScaleRef S;
  const PdhgState* __restrict__ st;
  BlockList bl;
  int kxprev_zero;
  double* __restrict__ partials;

  struct Regs {
    float sigma, theta;
    float yo[CHECK ? CAP : 1], kx[CHECK ? CAP : 1], kxe[CHECK ? CAP : 1];
    double acc0, acc1;
  };

  __device__ __forceinline__ float begin(Regs& r) const {
    r.sigma = st->sigma;
    r.theta = st->theta;
    r.acc0 = r.acc1 = 0.0;
    return r.sigma;
  }
  __device__ __forceinline__ float load(Regs& r, uint32_t e, int i) const {
    const float yv = y[e];
    const float k1 = gather_row(bl, e, x_new);
    const float k0 = kxprev_zero ? 0.f : gather_row(bl, e, x_old);
    const float ext = dual_extrapolate(r.theta, k1, k0);
    if (CHECK) {
      r.yo[i] = yv;
      r.kx[i] = k1;
      r.kxe[i] = ext;
    }
    return dual_prox_arg(yv, r.sigma, S.at(e), ext);
  }
  __device__ __forceinline__ void post(Regs& r, uint32_t e, int i, float yn) const {
    if (CHECK) {
      const float sq = sqrtf(S.at(e));
      const float z_hat = (r.yo[i] - yn) / (r.sigma * sq) + sq * r.kxe[i];
      const float diff = z_hat - sq * r.kx[i];
      r.acc0 += static_cast<double>(diff * diff);
      r.acc1 += static_cast<double>(z_hat * z_hat);
    }
  }
  __device__ __forceinline__ void finish(Regs& r) const {
    if (CHECK) {
      block_sum2(r.acc0, r.acc1);
      if (threadIdx.x == 0) { partials[2 * blockIdx.x] = r.acc0; partials[2 * blockIdx.x + 1] = r.acc1; }
    }
  }
};

#endif  // __CUDACC__

// Operands of one primal pass over the range of one prox (generic here, specialised in pb_stencil.cuh):
// x_out = prox_g(x - tau T K^T y).  kty_zero / ktyprev_zero take K^T y / K^T y_prev as 0 (the reference's
// quirks above); with `check` the pass also writes the dual residual sums to `partials`.  `halo` (slab mode, read by
// the specialised passes only) selects their slab variants when it has a neighbour.
struct PrimalPass {
  const float* x = nullptr;
  const float* y = nullptr;
  const float* y_prev = nullptr;      // check only
  ScaleRef T = {};
  const PdhgState* st = nullptr;
  bool kty_zero = false, ktyprev_zero = false, check = false;
  double* partials = nullptr;         // 2 doubles per CTA, check only
  unsigned partials_cap = 0;          // (a, b) pairs left at partials
  float* x_out = nullptr;
  const SlabHalo* halo = nullptr;
};

// Operands of one dual pass: y_out = prox_f*(y + sigma S ((1+theta) K x_new - theta K x_old)).  kxprev_zero
// takes K x_old as 0; with `check` the pass also writes the primal residual sums to `partials`.  `halo`: as above.
struct DualPass {
  const float* y = nullptr;
  const float* x_new = nullptr;
  const float* x_old = nullptr;
  ScaleRef S = {};
  const PdhgState* st = nullptr;
  bool kxprev_zero = false, check = false;
  double* partials = nullptr;         // 2 doubles per CTA, check only
  unsigned partials_cap = 0;          // (a, b) pairs left at partials
  float* y_out = nullptr;
  const SlabHalo* halo = nullptr;
};

// A residual-refresh pass writes one (a, b) pair per CTA at its partials: refuses a grid that would write past the
// `cap` pairs left there.
inline void check_partials_fit(bool check, unsigned grid, unsigned cap) {
  if (check && grid > cap)
    fail(PB_ERR_CUDA, "residual-refresh pass of " + std::to_string(grid) + " CTAs has room for only " +
                          std::to_string(cap) + " partial sums");
}

// Host-side launchers (pb_fused.cu); return the grid size.
unsigned fused_primal_launch(Context* ctx, const ProxDesc& d, const BlockList& bl, const PrimalPass& p);
unsigned fused_dual_launch(Context* ctx, const ProxDesc& d, const BlockList& bl, const DualPass& p);
unsigned fused_grid(Context* ctx, const ProxDesc& d);

}  // namespace pb
