// pb_stencil.cuh -- specialised fused PDHG passes for gradient operators in the planar layout.
//
// The generic fused kernel (pb_fused.cuh) interprets block/prox descriptors per element and
// spends several hundred instructions per pixel doing so; on B200 that makes a 44 B/pixel
// iteration instruction-bound (ncu: profiles/r1_generic_fused.md).  The kernels here fix the
// operator structure at compile time:
//
//   K = [ BlockGradient2D | BlockGradient3D ]  at row 0 / col 0, label_first = false
//       (+ optionally one identity block  f * I  below it, as in the lifted multilabel energy)
//
// and map threads to the image instead of to descriptor indices:
//   * a thread owns VEC (1 or 4) consecutive y of one column, read with 128-bit loads;
//   * (x, y, l) come from two multiply-high divisions per THREAD, not per element;
//   * the y-neighbour comes from the thread's own vector (+ one scalar load), the x- and
//     label-neighbours from aligned vector loads that hit L1/L2 (they are some other thread's
//     primary loads), so every array still crosses HBM exactly once per pass;
//   * the prox kind is a template parameter, the group lives in registers.
//
// Arithmetic (operation order, boundary handling, residual formulas) is identical to the generic
// fused pass and therefore to the reference:
//   forward  block_gradient2d.cu:25-78, block_gradient3d.cu:25-81 (Neumann in x, y; Dirichlet in l)
//   adjoint  block_gradient2d.cu:80-139, block_gradient3d.cu:83-150
//   primal / dual arguments and residuals  backend_pdhg.cu:38-120
#pragma once

#include "pb_backend.cuh"
#include "pb_comm.cuh"
#include "pb_crosssum.cuh"
#include "pb_fused.cuh"
#include "pb_prox.cuh"
#include "pb_reduce.cuh"

namespace pb {

// Residual-refresh launches of the ring kernel finish the iteration themselves: the last CTA to arrive (ticket)
// folds the per-CTA partial sums in index order, on slabs combines them across ranks through peer-mapped slots
// (cross_rank_sum4, pb_crosssum.cuh: identical bits on all ranks), and runs the step-size state machine
// (pdhg_update) -- no fold / all-reduce / finalize launches on the iteration path.  ticket == nullptr: the caller
// finalizes (NCCL staging mode).
struct RingFinish {
  unsigned* ticket = nullptr;
  PdhgState* state = nullptr;
  PdhgParams prm;
  unsigned long long iteration = 0;
  CrossSum cross;
};

// Operands of one launch of the ring kernel: the primal and the dual pass of one iteration (PrimalPass /
// DualPass in one).  With `check` it also reads y_prev and writes the dual (part_d) and primal (part_p)
// residual sums; `halo` selects the slab variants.
struct TilePass {
  const float* x = nullptr;
  const float* y = nullptr;
  const float* y_prev = nullptr;       // check only
  ScaleRef T = {}, S = {};             // uniform: only .val is read
  const PdhgState* st = nullptr;
  bool check = false;
  bool ktyprev_zero = true;            // check only
  double* part_d = nullptr;            // check only
  double* part_p = nullptr;
  unsigned part_cap = 0;               // check only: (a, b) pairs that fit at part_d and at part_p
  float* x_out = nullptr;
  float* y_out = nullptr;
  const RingHalo* halo = nullptr;      // slab mode
  const RingFinish* finish = nullptr;  // check only: the launch finalizes the iteration itself
  bool reverse = false;                // walk the tiles last to first (ignored in slab mode)
};

struct GradGeom {
  uint32_t nx = 0, ny = 0, L = 0, nxny = 0, plane = 0;
  uint32_t q = 0;                 // ny / VEC
  FastDiv div_q, div_nx, div_L;
  int has_id = 0;                 // identity block  id_factor * I  at rows [id_row, id_row + plane)
  uint32_t id_row = 0;
  float id_factor = 1.f;
  SlabHalo halo;                  // the pass's PrimalPass / DualPass::halo, all zero on a single GPU
};

constexpr int kStencilBlock = 128;

// Slab kernels map the edge column to threads [0, n_l * q) (n_l = L for per-voxel groups, 1 for
// per-pixel groups): the number of CTAs the last edge CTA waits for before it publishes the halo.
inline unsigned count_edge_ctas(uint32_t q, uint32_t n_l) {
  return (unsigned)(((size_t)q * n_l + kStencilBlock - 1) / kStencilBlock);
}

#ifdef __CUDACC__

template <int VEC> struct VecIO;
template <> struct VecIO<1> {
  static __device__ __forceinline__ void ld(const float* __restrict__ p, float (&o)[1]) { o[0] = *p; }
  static __device__ __forceinline__ void st(float* __restrict__ p, const float (&v)[1]) { *p = v[0]; }
};
template <> struct VecIO<4> {
  static __device__ __forceinline__ void ld(const float* __restrict__ p, float (&o)[4]) {
    const float4 t = *reinterpret_cast<const float4*>(p);
    o[0] = t.x; o[1] = t.y; o[2] = t.z; o[3] = t.w;
  }
  static __device__ __forceinline__ void st(float* __restrict__ p, const float (&v)[4]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
};

// ---- halo protocol (device side) ---------------------------------------------------------------------
// Edge threads spin (acquire, system scope) until the neighbour has published sequence `wait_seq`.
// Bounded: after ~2 s the kernel gives up, raises the error word and carries on with stale data so
// that a dead neighbour cannot hang the GPU.
__device__ __forceinline__ void halo_wait(const SlabHalo& h) {
  if (!h.wait_flag || h.wait_seq == 0) return;
  if (h.error && *reinterpret_cast<volatile int*>(h.error)) return;   // sticky: one timeout poisons the solve
  unsigned v;
  unsigned long long t0 = 0;
  for (unsigned spins = 0;; ++spins) {
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(h.wait_flag) : "memory");
    if ((int)(v - h.wait_seq) >= 0) break;
    if ((spins & 1023u) == 1023u) {
      unsigned long long now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      else if (now - t0 > 2000000000ull) { if (h.error) atomicExch(h.error, 1); break; }
    }
  }
}

// Called by every thread of the CTA at the end of a pass.  Edge threads fence their remote stores,
// the CTA's thread 0 counts the CTA in, and the last edge CTA publishes the sequence number in the
// neighbour's memory (release, system scope) -- by then every halo store AND every halo load of
// this launch has been performed, which is what makes two ping-pong slots sufficient.
__device__ __forceinline__ void halo_signal(const SlabHalo& h, bool edge_thread) {
  if (!h.done_counter) return;                                 // uniform: single GPU or NCCL staging
  if (edge_thread) __threadfence_system();
  const int any = __syncthreads_or(edge_thread ? 1 : 0);
  if (any && threadIdx.x == 0) {
    const unsigned prev = atomicAdd(h.done_counter, 1u);
    if (prev + 1 == h.n_edge_ctas) {
      atomicExch(h.done_counter, 0u);
      __threadfence_system();
      if (h.signal_flag)
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(h.signal_flag), "r"(h.signal_seq) : "memory");
    }
  }
}

template <int VEC>
__device__ __forceinline__ void load_scale(const ScaleRef& s, uint32_t e, float (&o)[VEC]) {
  if (s.ptr) {
    VecIO<VEC>::ld(s.ptr + e, o);
  } else {
#pragma unroll
    for (int j = 0; j < VEC; ++j) o[j] = s.val;
  }
}

// forward differences of u at idx .. idx+VEC-1 (same column x, label l)
template <int VEC, bool THREE_D, bool SLAB>
__device__ __forceinline__ void grad_fwd(const GradGeom& g, const float* __restrict__ u,
                                         const float* __restrict__ u_halo, uint32_t idx,
                                         uint32_t x, uint32_t y0, uint32_t l, float (&gx)[VEC],
                                         float (&gy)[VEC], float (&gl)[VEC]) {
  float c[VEC], n[VEC];
  VecIO<VEC>::ld(u + idx, c);
  if (x < g.nx - 1) {
    VecIO<VEC>::ld(u + idx + g.ny, n);
#pragma unroll
    for (int j = 0; j < VEC; ++j) gx[j] = n[j] - c[j];
  } else if (SLAB && g.halo.has_right) {
    // slab edge: column x+1 lives on the right neighbour
    VecIO<VEC>::ld(u_halo + y0 + l * g.ny, n);
#pragma unroll
    for (int j = 0; j < VEC; ++j) gx[j] = n[j] - c[j];
  } else {
#pragma unroll
    for (int j = 0; j < VEC; ++j) gx[j] = 0.f;
  }
#pragma unroll
  for (int j = 0; j + 1 < VEC; ++j) gy[j] = c[j + 1] - c[j];
  gy[VEC - 1] = (y0 + VEC < g.ny) ? u[idx + VEC] - c[VEC - 1] : 0.f;
  if (THREE_D) {
    if (l < g.L - 1) {
      VecIO<VEC>::ld(u + idx + g.nxny, n);
#pragma unroll
      for (int j = 0; j < VEC; ++j) gl[j] = n[j] - c[j];
    } else {
#pragma unroll
      for (int j = 0; j < VEC; ++j) gl[j] = -c[j];
    }
  }
}

// (K^T p) at idx .. idx+VEC-1 : minus divergence (+ identity rows)
template <int VEC, bool THREE_D, bool HAS_ID, bool SLAB>
__device__ __forceinline__ void grad_adj(const GradGeom& g, const float* __restrict__ p,
                                         const float* __restrict__ p_halo, uint32_t idx,
                                         uint32_t x, uint32_t y0, uint32_t l, float (&out)[VEC]) {
  const float* __restrict__ p1 = p;
  const float* __restrict__ p2 = p + g.plane;
  float a[VEC], divx[VEC], divy[VEC], o[VEC];
  if (x < g.nx - 1 || (SLAB && g.halo.has_right)) {
    VecIO<VEC>::ld(p1 + idx, divx);
  } else {
#pragma unroll
    for (int j = 0; j < VEC; ++j) divx[j] = 0.f;
  }
  if (x > 0) {
    VecIO<VEC>::ld(p1 + idx - g.ny, a);
#pragma unroll
    for (int j = 0; j < VEC; ++j) divx[j] -= a[j];
  } else if (SLAB && g.halo.has_left) {
    // slab edge: column x-1 of the x-component lives on the left neighbour
    VecIO<VEC>::ld(p_halo + y0 + l * g.ny, a);
#pragma unroll
    for (int j = 0; j < VEC; ++j) divx[j] -= a[j];
  }
  VecIO<VEC>::ld(p2 + idx, o);
#pragma unroll
  for (int j = 0; j < VEC; ++j) divy[j] = o[j];
  if (y0 + VEC == g.ny) divy[VEC - 1] = 0.f;              // y = ny-1
#pragma unroll
  for (int j = 1; j < VEC; ++j) divy[j] -= o[j - 1];
  if (y0 > 0) divy[0] -= p2[idx - 1];
  if (THREE_D) {
    const float* __restrict__ p3 = p + 2u * (size_t)g.plane;
    float d[VEC];
    VecIO<VEC>::ld(p3 + idx, d);
    if (l > 0) {
      VecIO<VEC>::ld(p3 + idx - g.nxny, a);
#pragma unroll
      for (int j = 0; j < VEC; ++j) d[j] -= a[j];
    }
#pragma unroll
    for (int j = 0; j < VEC; ++j) out[j] = -(divx[j] + divy[j] + d[j]);
  } else {
#pragma unroll
    for (int j = 0; j < VEC; ++j) out[j] = -(divx[j] + divy[j]);
  }
  if (HAS_ID) {
    VecIO<VEC>::ld(p + g.id_row + idx, a);
#pragma unroll
    for (int j = 0; j < VEC; ++j) out[j] = __fadd_rn(out[j], __fmul_rn(a[j], g.id_factor));
  }
}

// true when every coefficient except b (index 1) is a scalar: the common "data term" shape
// c*f(a x - b) with a per-pixel b (the image) and scalar weights
__device__ __forceinline__ bool coeffs_scalar_except_b(const CoeffRef& c) {
  return !c.ptr[0] && !c.ptr[2] && !c.ptr[3] && !c.ptr[4] && !c.ptr[5] && !c.ptr[6];
}

// ---- primal pass:  x+ = prox_g( x - tau T K^T y ) ----------------------------------------------------
//  CAPL == 1 : thread = (y-vector, x, l); the prox group is one element (Elem1D / Zero), p.count = plane
//  CAPL  > 1 : thread = (y-vector, x);    the prox group spans the L <= CAPL labels of a pixel, planar,
//              p.count = nx*ny, p.dim = L  (simplex over labels)
//  TUNI: the preconditioner T is one scalar (always true for pure gradient operators), which lets
//  the compiler hoist every step-size expression out of the per-lane code.
template <int VEC, int CAPL, int KIND, int FN, bool THREE_D, bool HAS_ID, bool CHECK, bool TUNI, bool SLAB>
__device__ __forceinline__ bool grad_primal_body(
    const GradGeom& g, const ProxDesc& p, const float* __restrict__ x, const float* __restrict__ y,
    const float* __restrict__ y_prev, const ScaleRef& T, const float tau, const int kty_zero,
    const int ktyprev_zero, float* __restrict__ x_out, const uint32_t t, double& acc0, double& acc1) {
  uint32_t xl, yv, l0 = 0, xx;
  g.div_q.divmod(t, xl, yv);
  // slab kernels put x slowest so that the edge column (x = 0) is the FIRST q*L threads of the grid:
  // its halo goes out, and the neighbour is signalled, at the start of the pass
  if (CAPL == 1) { if (SLAB) g.div_L.divmod(xl, xx, l0); else g.div_nx.divmod(xl, l0, xx); } else xx = xl;
  const uint32_t y0 = yv * VEC;
  const uint32_t pix = y0 + xx * g.ny;
  const uint32_t nl = CAPL == 1 ? 1u : g.L;
  // slab edge towards the left neighbour: its y halo must have arrived before K^T y is gathered
  const bool edge = SLAB && g.halo.has_left && xx == 0;
  if (SLAB && edge && !(kty_zero && (!CHECK || ktyprev_zero))) halo_wait(g.halo);

  float arg[CAPL][VEC], td[CAPL][VEC];
#pragma unroll
  for (int li = 0; li < CAPL; ++li) {
#pragma unroll
    for (int j = 0; j < VEC; ++j) { arg[li][j] = 0.f; td[li][j] = TUNI ? T.val : 1.f; }
    if (li < (int)nl) {
      const uint32_t l = l0 + li;
      const uint32_t idx = pix + l * g.nxny;
      float xo[VEC], k[VEC];
      VecIO<VEC>::ld(x + idx, xo);
      if (kty_zero) {
#pragma unroll
        for (int j = 0; j < VEC; ++j) k[j] = 0.f;
      } else {
        grad_adj<VEC, THREE_D, HAS_ID, SLAB>(g, y, g.halo.in_a, idx, xx, y0, l, k);
      }
      if (!TUNI) VecIO<VEC>::ld(T.ptr + idx, td[li]);
#pragma unroll
      for (int j = 0; j < VEC; ++j) arg[li][j] = primal_prox_arg(xo[j], tau, td[li][j], k[j]);
    }
  }
  // prox, one lane (= one group) at a time
  const uint32_t tx0 = CAPL == 1 ? pix + l0 * g.nxny : pix;
  if (KIND == kProxElem1D && CAPL == 1 && TUNI && !p.moreau && coeffs_scalar_except_b(p.coeffs)) {
    // scalar weights: everything but b is loop invariant across the lanes
    Coeffs7 c;
#pragma unroll
    for (int k = 0; k < 7; ++k) c.v[k] = p.coeffs.val[k];
    float bv[VEC];
    if (p.coeffs.ptr[1]) {
      VecIO<VEC>::ld(p.coeffs.ptr[1] + tx0, bv);
    } else {
#pragma unroll
      for (int j = 0; j < VEC; ++j) bv[j] = p.coeffs.val[1];
    }
    const int fn = FN >= 0 ? FN : p.fn;
    if (coeffs_simple(c) && c.v[2] != 0.f) {
      const float tau_eff = effective_tau(tau, T.val, false);
#pragma unroll
      for (int j = 0; j < VEC; ++j)
        arg[0][j] = scaled_fun_prox_simple(fn, arg[0][j], tau_eff, bv[j], c.v[2], c.v[5], c.v[6]);
    } else {
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        c.v[1] = bv[j];
        arg[0][j] = elem1d_apply(fn, arg[0][j], tau, T.val, false, c);
      }
    }
  } else {
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      float v[CAPL], tdl[CAPL];
#pragma unroll
      for (int li = 0; li < CAPL; ++li) { v[li] = arg[li][j]; tdl[li] = td[li][j]; }
      group_apply<CAPL, KIND, FN>(p, tx0 + j, v, tdl, tau, false);
#pragma unroll
      for (int li = 0; li < CAPL; ++li) arg[li][j] = v[li];
    }
  }
#pragma unroll
  for (int li = 0; li < CAPL; ++li) {
    if (li < (int)nl) {
      const uint32_t l = l0 + li;
      const uint32_t idx = pix + l * g.nxny;
      VecIO<VEC>::st(x_out + idx, arg[li]);
      if (SLAB && edge) VecIO<VEC>::st(g.halo.out + y0 + l * g.ny, arg[li]);   // new column 0 -> left neighbour
      if (CHECK) {
        // dual residual (backend_pdhg.cu:73-94); operands are re-read (L1/L2 resident) rather
        // than kept live across the prox
        float xo[VEC], k[VEC], kp[VEC];
        VecIO<VEC>::ld(x + idx, xo);
        if (kty_zero) {
#pragma unroll
          for (int j = 0; j < VEC; ++j) k[j] = 0.f;
        } else {
          grad_adj<VEC, THREE_D, HAS_ID, SLAB>(g, y, g.halo.in_a, idx, xx, y0, l, k);
        }
        if (ktyprev_zero) {
#pragma unroll
          for (int j = 0; j < VEC; ++j) kp[j] = 0.f;
        } else {
          grad_adj<VEC, THREE_D, HAS_ID, SLAB>(g, y_prev, g.halo.in_b, idx, xx, y0, l, kp);
        }
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          const float sq = sqrtf(td[li][j]);
          const float w_hat = (xo[j] - arg[li][j]) / (tau * sq) - sq * kp[j];
          const float diff = w_hat + sq * k[j];
          acc0 += static_cast<double>(diff * diff);
          acc1 += static_cast<double>(w_hat * w_hat);
        }
      }
    }
  }
  return edge;
}

template <int VEC, int CAPL, int KIND, int FN, bool THREE_D, bool HAS_ID, bool CHECK, bool SLAB>
__global__ void __launch_bounds__(kStencilBlock) grad_primal_kernel(
    const GradGeom g, const ProxDesc p, const float* __restrict__ x, const float* __restrict__ y,
    const float* __restrict__ y_prev, const ScaleRef T, const PdhgState* __restrict__ st,
    const int kty_zero, const int ktyprev_zero, double* __restrict__ partials, float* __restrict__ x_out) {
  const float tau = st->tau;
  double acc0 = 0.0, acc1 = 0.0;
  const uint32_t total = g.q * g.nx * (CAPL == 1 ? g.L : 1u);
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  bool edge = false;
  if (t < total) {
    if (T.ptr)
      edge = grad_primal_body<VEC, CAPL, KIND, FN, THREE_D, HAS_ID, CHECK, false, SLAB>(
          g, p, x, y, y_prev, T, tau, kty_zero, ktyprev_zero, x_out, t, acc0, acc1);
    else
      edge = grad_primal_body<VEC, CAPL, KIND, FN, THREE_D, HAS_ID, CHECK, true, SLAB>(
          g, p, x, y, y_prev, T, tau, kty_zero, ktyprev_zero, x_out, t, acc0, acc1);
  }
  if (SLAB) halo_signal(g.halo, edge);
  if (CHECK) {
    block_sum2(acc0, acc1);
    if (threadIdx.x == 0) { partials[2 * blockIdx.x] = acc0; partials[2 * blockIdx.x + 1] = acc1; }
  }
}

// Norm2 prox of VEC groups held in registers, scalar weights (elem_operation_norm2.hpp:39-88):
// res_i = ((f_prox(a(|v| - d tau)/(1 + tau e) - b, .) + b)/a) * v_i / |v|.  The per-component
// division by the shared norm uses div_shared.
template <int VEC, int CAP, bool SIMPLE>
__device__ __forceinline__ void norm2_lanes(const int fn, float (&arg)[CAP][VEC], const Coeffs7& c,
                                            const float tau_eff) {
#pragma unroll
  for (int j = 0; j < VEC; ++j) {
    float sq = 0.f;
#pragma unroll
    for (int s = 0; s < CAP; ++s) sq += arg[s][j] * arg[s][j];
    if (sq > 0.f) {
      const float norm = sqrtf(sq);
      const float r = SIMPLE ? scaled_fun_prox_simple(fn, norm, tau_eff, c.v[1], c.v[2], c.v[5], c.v[6])
                             : scaled_fun_prox(fn, norm, tau_eff, c);
      const float rn = 1.f / norm;
#pragma unroll
      for (int s = 0; s < CAP; ++s) arg[s][j] = div_shared(__fmul_rn(r, arg[s][j]), norm, rn);
    } else {
#pragma unroll
      for (int s = 0; s < CAP; ++s) arg[s][j] = 0.f;
    }
  }
}

// ---- dual pass on the gradient rows:  y+ = prox_f*( y + sigma S ((1+theta) K x+ - theta K x) ) -------
//  prox = Norm2 family (optionally through Moreau), planar:
//  CAPL == 1 : thread = (y-vector, x, l); group = the NCOMP components of one voxel,
//              p.count = plane, p.dim = NCOMP
//  CAPL  > 1 : thread = (y-vector, x);    group = NCOMP * L components of one pixel (L <= CAPL),
//              p.count = nx*ny, p.dim = NCOMP * L, component i = c*L + l
template <int VEC, int CAPL, int FN, bool THREE_D, bool CHECK, bool SUNI, bool SLAB>
__device__ __forceinline__ bool grad_dual_body(
    const GradGeom& g, const ProxDesc& p, const float* __restrict__ y, const float* __restrict__ xn,
    const float* __restrict__ xo, const ScaleRef& S, const float sigma, const float theta,
    const int kxprev_zero, float* __restrict__ y_out, const uint32_t t, double& acc0, double& acc1) {
  constexpr int NCOMP = THREE_D ? 3 : 2;
  constexpr int CAP = NCOMP * CAPL;
  uint32_t xl, yv, l0 = 0, xx;
  g.div_q.divmod(t, xl, yv);
  // slab kernels walk x from the right so that the edge column (x = nx-1) is the first q*L threads
  if (CAPL == 1) { if (SLAB) g.div_L.divmod(xl, xx, l0); else g.div_nx.divmod(xl, l0, xx); } else xx = xl;
  if (SLAB) xx = g.nx - 1 - xx;
  const uint32_t y0 = yv * VEC;
  const uint32_t pix = y0 + xx * g.ny;
  const uint32_t nl = CAPL == 1 ? 1u : g.L;
  // slab edge towards the right neighbour: its x halo must have arrived before K x is gathered
  const bool edge = SLAB && g.halo.has_right && xx == g.nx - 1;
  if (SLAB && edge) halo_wait(g.halo);

  // slot (c, li) -> c*CAPL + li ; unused label slots stay 0 (they do not change a 2-norm)
  float arg[CAP][VEC], td[SUNI ? 1 : CAP][VEC];
#pragma unroll
  for (int s = 0; s < CAP; ++s) {
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      arg[s][j] = 0.f;
      if (!SUNI) td[s][j] = 1.f;
    }
  }
  if (SUNI) {
#pragma unroll
    for (int j = 0; j < VEC; ++j) td[0][j] = S.val;
  }
#pragma unroll
  for (int li = 0; li < CAPL; ++li) {
    if (li < (int)nl) {
      const uint32_t l = l0 + li;
      const uint32_t idx = pix + l * g.nxny;
      float k1[NCOMP][VEC], k0[NCOMP][VEC];
      grad_fwd<VEC, THREE_D, SLAB>(g, xn, g.halo.in_a, idx, xx, y0, l, k1[0], k1[1], k1[NCOMP - 1]);
      if (kxprev_zero) {
#pragma unroll
        for (int c = 0; c < NCOMP; ++c)
#pragma unroll
          for (int j = 0; j < VEC; ++j) k0[c][j] = 0.f;
      } else {
        grad_fwd<VEC, THREE_D, SLAB>(g, xo, g.halo.in_b, idx, xx, y0, l, k0[0], k0[1], k0[NCOMP - 1]);
      }
#pragma unroll
      for (int c = 0; c < NCOMP; ++c) {
        const uint32_t e = c * g.plane + idx;
        const int s = c * CAPL + li;
        float yo[VEC];
        VecIO<VEC>::ld(y + e, yo);
        if (!SUNI) VecIO<VEC>::ld(S.ptr + e, td[s]);
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          const float ext = dual_extrapolate(theta, k1[c][j], k0[c][j]);
          arg[s][j] = dual_prox_arg(yo[j], sigma, td[SUNI ? 0 : s][j], ext);
        }
      }
    }
  }
  const uint32_t tx0 = CAPL == 1 ? pix + l0 * g.nxny : pix;
  const int fn = FN >= 0 ? FN : p.fn;
  bool scalar_coeffs = SUNI && !p.moreau;
#pragma unroll
  for (int k = 0; k < 7; ++k) scalar_coeffs = scalar_coeffs && !p.coeffs.ptr[k];
  if (scalar_coeffs) {
    // all weights scalar: the step and every coefficient product are lane invariant
    Coeffs7 c;
#pragma unroll
    for (int k = 0; k < 7; ++k) c.v[k] = p.coeffs.val[k];
    const float tau_eff = effective_tau(sigma, S.val, false);
    if (coeffs_simple(c))
      norm2_lanes<VEC, CAP, true>(fn, arg, c, tau_eff);
    else
      norm2_lanes<VEC, CAP, false>(fn, arg, c, tau_eff);
  } else {
    ProxDesc pd = p;
    pd.dim = CAP;
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      float v[CAP], tdl[CAP];
#pragma unroll
      for (int s = 0; s < CAP; ++s) { v[s] = arg[s][j]; tdl[s] = td[SUNI ? 0 : s][j]; }
      group_apply<CAP, kProxNorm2, FN>(pd, tx0 + j, v, tdl, sigma, false);
#pragma unroll
      for (int s = 0; s < CAP; ++s) arg[s][j] = v[s];
    }
  }
#pragma unroll
  for (int li = 0; li < CAPL; ++li) {
    if (li < (int)nl) {
      const uint32_t l = l0 + li;
      const uint32_t idx = pix + l * g.nxny;
      float k1[NCOMP][VEC], k0[NCOMP][VEC];
      if (CHECK) {
        grad_fwd<VEC, THREE_D, SLAB>(g, xn, g.halo.in_a, idx, xx, y0, l, k1[0], k1[1], k1[NCOMP - 1]);
        if (kxprev_zero) {
#pragma unroll
          for (int c = 0; c < NCOMP; ++c)
#pragma unroll
            for (int j = 0; j < VEC; ++j) k0[c][j] = 0.f;
        } else {
          grad_fwd<VEC, THREE_D, SLAB>(g, xo, g.halo.in_b, idx, xx, y0, l, k0[0], k0[1], k0[NCOMP - 1]);
        }
      }
#pragma unroll
      for (int c = 0; c < NCOMP; ++c) {
        const uint32_t e = c * g.plane + idx;
        const int s = c * CAPL + li;
        VecIO<VEC>::st(y_out + e, arg[s]);
        if (SLAB && c == 0 && edge) VecIO<VEC>::st(g.halo.out + y0 + l * g.ny, arg[s]);  // last gx column -> right
        if (CHECK) {
          // primal residual (backend_pdhg.cu:97-120)
          float yo[VEC];
          VecIO<VEC>::ld(y + e, yo);
#pragma unroll
          for (int j = 0; j < VEC; ++j) {
            const float ext = dual_extrapolate(theta, k1[c][j], k0[c][j]);
            const float sq = sqrtf(td[SUNI ? 0 : s][j]);
            const float z_hat = (yo[j] - arg[s][j]) / (sigma * sq) + sq * ext;
            const float diff = z_hat - sq * k1[c][j];
            acc0 += static_cast<double>(diff * diff);
            acc1 += static_cast<double>(z_hat * z_hat);
          }
        }
      }
    }
  }
  return edge;
}

template <int VEC, int CAPL, int FN, bool THREE_D, bool CHECK, bool SLAB>
__global__ void __launch_bounds__(kStencilBlock) grad_dual_norm2_kernel(
    const GradGeom g, const ProxDesc p, const float* __restrict__ y, const float* __restrict__ xn,
    const float* __restrict__ xo, const ScaleRef S, const PdhgState* __restrict__ st, const int kxprev_zero,
    double* __restrict__ partials, float* __restrict__ y_out) {
  const float sigma = st->sigma, theta = st->theta;
  double acc0 = 0.0, acc1 = 0.0;
  const uint32_t total = g.q * g.nx * (CAPL == 1 ? g.L : 1u);
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  bool edge = false;
  if (t < total) {
    if (S.ptr)
      edge = grad_dual_body<VEC, CAPL, FN, THREE_D, CHECK, false, SLAB>(g, p, y, xn, xo, S, sigma, theta,
                                                                        kxprev_zero, y_out, t, acc0, acc1);
    else
      edge = grad_dual_body<VEC, CAPL, FN, THREE_D, CHECK, true, SLAB>(g, p, y, xn, xo, S, sigma, theta,
                                                                       kxprev_zero, y_out, t, acc0, acc1);
  }
  if (SLAB) halo_signal(g.halo, edge);
  if (CHECK) {
    block_sum2(acc0, acc1);
    if (threadIdx.x == 0) { partials[2 * blockIdx.x] = acc0; partials[2 * blockIdx.x + 1] = acc1; }
  }
}

// ---- dual pass on identity rows:  K x = f * x  (no stencil), any register-resident leaf prox ----------
template <int CAP, bool CHECK>
struct IdentityDualSource {
  const float* __restrict__ y;
  const float* __restrict__ x_new;    // already offset so that row e reads x[e - id_row]
  const float* __restrict__ x_old;
  ScaleRef S;
  const PdhgState* __restrict__ st;
  float factor;
  uint32_t id_row;
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
    const float k1 = __fmul_rn(x_new[e - id_row], factor);
    const float k0 = kxprev_zero ? 0.f : __fmul_rn(x_old[e - id_row], factor);
    const float ext = dual_extrapolate(r.theta, k1, k0);
    if (CHECK) { r.yo[i] = yv; r.kx[i] = k1; r.kxe[i] = ext; }
    return dual_prox_arg(yv, r.sigma, S.at(e), ext);
  }
  // four consecutive rows at once (prox_pass_pairs4_kernel; uniform S, no residual terms)
  __device__ __forceinline__ void load4(Regs& r, uint32_t e, float (&out)[4]) const {
    const float4 yv = *reinterpret_cast<const float4*>(y + e);
    const float4 xn = *reinterpret_cast<const float4*>(x_new + (e - id_row));
    float4 xo = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!kxprev_zero) xo = *reinterpret_cast<const float4*>(x_old + (e - id_row));
    const float yy[4] = {yv.x, yv.y, yv.z, yv.w}, n4[4] = {xn.x, xn.y, xn.z, xn.w}, o4[4] = {xo.x, xo.y, xo.z, xo.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float k1 = __fmul_rn(n4[q], factor);
      const float k0 = kxprev_zero ? 0.f : __fmul_rn(o4[q], factor);
      out[q] = dual_prox_arg(yy[q], r.sigma, S.val, dual_extrapolate(r.theta, k1, k0));
    }
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

// ---- host side: pattern matching + launch (pb_stencil.cu) -----------------------------------------

struct StencilPlan {
  bool ok = false;            // operator matches  [gradient (+ identity)]
  bool three_d = false;
  GradGeom geom;              // q / div_q filled per launch (depends on VEC)
};

// Recognises the operator structure; `blocks` are the problem's non-zero blocks.
StencilPlan plan_stencil(const std::vector<std::shared_ptr<Block>>& blocks, size_t nrows, size_t ncols);

// Does a specialised pass cover prox `d` of the plan's operator?  0 if not (the generic fused pass runs it), otherwise
// the largest grid any variant of that pass launches for it, i.e. the most (a, b) partial pairs it writes.  Which
// variant runs is decided per launch, from the operands' alignment and the iteration.
unsigned stencil_primal_cover(const StencilPlan& plan, const ProxDesc& d);
unsigned stencil_dual_cover(const Context* ctx, const StencilPlan& plan, const ProxDesc& d);
// Each returns 0 when the pass is not covered, otherwise the number of CTAs launched (= partial pairs written).
unsigned stencil_primal_launch(Context* ctx, const StencilPlan& plan, const ProxDesc& d, const PrimalPass& p);
unsigned stencil_dual_launch(Context* ctx, const StencilPlan& plan, const ProxDesc& d, const DualPass& p);

// ---- whole iteration as one tiled pass (pb_tile.cu) ---------------------------------------------
// Can the one-pass ring kernel run every iteration after the first (slab: its halo variants)?
bool tile_ring_available(const StencilPlan& plan, const std::vector<ProxDesc>& gd, const std::vector<ProxDesc>& fd,
                         ScaleRef T, ScaleRef S, bool slab);
// its grid, i.e. the (a, b) partial pairs a residual-refresh launch writes to each of part_d and part_p
unsigned tile_ring_grid(const Context* ctx, const StencilPlan& plan);
// one iteration as one tiled pass; returns the number of (a, b) partial pairs written to each of part_d and
// part_p (0 unless p.check); raises PB_ERR_CUDA if the ring kernel cannot be launched
unsigned tile_iteration_launch(Context* ctx, const StencilPlan& plan, const ProxDesc& pg, const ProxDesc& pf,
                               const TilePass& p);
unsigned tile_ring_trace_read(unsigned long long* h_out, unsigned n);      // PB_RING_TRACE experiments

}  // namespace pb
