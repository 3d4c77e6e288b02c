// pb_admm.cu -- BackendADMM: graph-projection ADMM with an inexact CGLS projection.
//
// Reference: BackendADMM<T>::Initialize / PerformIteration / current_solution
// (src/backend/backend_admm.cu:285-352, 354-665, 669-741), GemvPrecondK (:198-272) and
// cgls::Solve (include/prost/cgls.hpp:222-371).
//
// The reference runs one outer iteration as ~25 thrust passes plus, per CG step, two operator
// applies wrapped in three element-wise passes each, six cuBLAS/thrust vector operations, four
// reductions and seven cudaDeviceSynchronize() calls, because every CG scalar travels through the
// host.  Here
//   * all CG scalars (gamma, alpha, beta, the norms, the convergence verdict) live in a CgState
//     struct in device memory; reductions are per-thread double -> warp shuffle -> one partial per
//     CTA, folded in index order by the last CTA to arrive (ticket), which then also advances the
//     scalar recurrences.  A whole outer iteration is enqueued without a single host round trip;
//   * when CG converges early the remaining enqueued steps see CgState::done and return at once
//     (the operator-apply kernels observe the same flag through Context::skip_flag);
//   * the element-wise work of GemvPrecondK, the axpys, the vector copies and the norm of every
//     vector are fused: one CG step is 4 element-wise kernels + 2 operator applies;
//   * rho only changes on residual iterations, where Solver::Solve needs the residuals on the host
//     anyway, so the residual-balancing state machine (:628-660) stays on the host.
// Arithmetic follows the reference expression by expression in float with double CG scalars
// (cgls.hpp:170-189, 241), including the GemvPrecondK factorisation (beta/(alpha*sqrt(S))) * y ...
// alpha*sqrt(S)*y, so iterates agree with the reference to rounding (summation order inside the
// SpMV / GEMV differs from cuSPARSE / cuBLAS).
#include <algorithm>
#include <cmath>
#include <iostream>
#include <limits>

#include "pb_backend.cuh"
#include "pb_comm.cuh"
#include "pb_crosssum.cuh"
#include "pb_reduce.cuh"

namespace pb {

namespace {

// Scalars of one cgls::Solve call (cgls.hpp:238-241) + control flags.
struct CgState {
  double gamma, normp, normq, norms, norms0, normx, xmax;
  float alpha, neg_alpha, beta;
  int done;         // loop left: converged (:354) or flag set before the loop (:287-288)
  int skip_init;    // normx == 0: "r = b - A x" is not evaluated (:250-257)
  int indefinite;
  int k;            // CG steps taken
  unsigned ticket;
};

// CTA partial -> global partial; the last CTA to arrive folds all partials in index order.
// Returns true in thread 0 of that CTA with (a, b) = totals.  All threads must call.
// `cross` (row-sharded ADMM): sums over the m-side rows are partial per rank; the folding thread then combines them
// through peer-mapped slots (pb_crosssum.cuh), so the scalar recurrences stay on the device and identical on all ranks.
__device__ __forceinline__ bool reduce_last(double& a, double& b, double* __restrict__ partials,
                                            unsigned* ticket, const CrossSum* cross = nullptr) {
  __shared__ int s_last;
  block_sum2(a, b);
  if (threadIdx.x == 0) {
    __stcg(partials + 2 * blockIdx.x, a);
    __stcg(partials + 2 * blockIdx.x + 1, b);
    __threadfence();
    s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1) ? 1 : 0;
  }
  __syncthreads();
  if (!s_last) return false;
  __threadfence();
  double fa = 0.0, fb = 0.0;
  for (unsigned i = threadIdx.x; i < gridDim.x; i += blockDim.x) {
    fa += __ldcg(partials + 2 * i);
    fb += __ldcg(partials + 2 * i + 1);
  }
  block_sum2(fa, fb);
  if (threadIdx.x == 0 && cross) {
    double v[4] = {fa, fb, 0.0, 0.0};
    cross_rank_sum4(*cross, v);
    fa = v[0];
    fb = v[1];
  }
  a = fa;
  b = fb;
  if (threadIdx.x == 0) *ticket = 0;
  return threadIdx.x == 0;
}

#define PB_GRID_STRIDE(i, n) \
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < (n); i += (size_t)gridDim.x * blockDim.x)

// ---- outer iteration, part 1 (backend_admm.cu:357-401) ------------------------------------------
// temp1 = (alpha x_half + (1-alpha) x_proj + x_dual) / sqrt(T)        temp1_functor :52-66
// temp2 = sqrt(S) (z_half + z_dual);  b = z_dual = temp2              temp2_functor :68-79, :394
// x_proj = temp3[0:n] (warm start :398);  s = x_proj (cgls.hpp:246);  |x|^2
// then the element-wise head of gemv('n', -1, temp1, 1, b):  temp3 = sqrt(T) temp1,
// b = (1 / (-1 sqrt(S))) b                                            gemv_functor1/2 :143-165
__global__ void __launch_bounds__(kBlock) admm_begin_kernel(
    size_t n, size_t m, float alpha, ScaleRef T, ScaleRef S, const float* __restrict__ x_half,
    float* __restrict__ x_proj, float* __restrict__ x_dual /* = cg s */, const float* __restrict__ z_half,
    float* __restrict__ z_dual /* = b */, float* __restrict__ temp1, float* __restrict__ temp2,
    float* __restrict__ temp3, CgState* cg, double* partials) {
  double acc = 0.0, unused = 0.0;
  const size_t len = n > m ? n : m;
  PB_GRID_STRIDE(i, len) {
    if (i < n) {
      const float st = sqrtf(T.at((uint32_t)i));
      const float t1 = (alpha * x_half[i] + (1 - alpha) * x_proj[i] + x_dual[i]) / st;
      temp1[i] = t1;
      const float x0 = temp3[i];
      x_proj[i] = x0;
      x_dual[i] = x0;
      acc += static_cast<double>(x0) * static_cast<double>(x0);
      temp3[i] = st * t1;
    }
    if (i < m) {
      const float ss = sqrtf(S.at((uint32_t)i));
      const float t2 = ss * (z_half[i] + z_dual[i]);
      temp2[i] = t2;
      z_dual[i] = (1.f / (-1.f * ss)) * t2;
    }
  }
  if (reduce_last(acc, unused, partials, &cg->ticket)) {
    cg->normx = sqrt(acc);
    cg->skip_init = (cg->normx > 0.) ? 0 : 1;
    cg->done = 0;
    cg->indefinite = 0;
    cg->k = 0;
  }
}

// tail of gemv('n', -1, temp1, 1, b): b = -1 sqrt(S) b (gemv_functor3 :167-180); r = b
// (cgls.hpp:245); if |x| > 0 the head of gemv('n', -1, x, 1, r): temp3 = sqrt(T) x,
// r = (1 / (-1 sqrt(S))) r
__global__ void __launch_bounds__(kBlock) admm_rhs_kernel(size_t n, size_t m, ScaleRef T, ScaleRef S,
                                                          const float* __restrict__ x,
                                                          float* __restrict__ b, float* __restrict__ r,
                                                          float* __restrict__ temp3,
                                                          const CgState* __restrict__ cg) {
  const bool skip = cg->skip_init != 0;
  const size_t len = n > m ? n : m;
  PB_GRID_STRIDE(i, len) {
    if (i < m) {
      const float ss = sqrtf(S.at((uint32_t)i));
      const float bv = (-1.f * ss) * b[i];
      b[i] = bv;
      r[i] = skip ? bv : (1.f / (-1.f * ss)) * bv;
    }
    if (i < n && !skip) temp3[i] = sqrtf(T.at((uint32_t)i)) * x[i];
  }
}

// tail of r = b - A x (if evaluated): r = -1 sqrt(S) r; then the head of
// gemv('t', 1, r, -shift, s):  temp3 = sqrt(S) r,  s = (-shift / (1 sqrt(T))) s
__global__ void __launch_bounds__(kBlock) cg_adjoint_head_kernel(size_t n, size_t m, ScaleRef T, ScaleRef S,
                                                                 float neg_shift, float* __restrict__ r,
                                                                 float* __restrict__ s,
                                                                 float* __restrict__ temp3,
                                                                 const CgState* __restrict__ cg) {
  const bool skip = cg->skip_init != 0;
  const size_t len = n > m ? n : m;
  PB_GRID_STRIDE(i, len) {
    if (i < m) {
      const float ss = sqrtf(S.at((uint32_t)i));
      float rv = r[i];
      if (!skip) { rv = (-1.f * ss) * rv; r[i] = rv; }
      temp3[i] = ss * rv;
    }
    if (i < n) s[i] = (neg_shift / (1.f * sqrtf(T.at((uint32_t)i)))) * s[i];
  }
}

// tail of the first gemv('t'): s = 1 sqrt(T) s; p = s (cgls.hpp:269); |s|; head of the first
// gemv('n', 1, p, 0, q): temp3 = sqrt(T) p.  Finalize :271-288.
__global__ void __launch_bounds__(kBlock) cg_init_tail_kernel(size_t n, ScaleRef T, float* __restrict__ s,
                                                              float* __restrict__ p,
                                                              float* __restrict__ temp3, CgState* cg,
                                                              double* partials, double k_eps) {
  double acc = 0.0, unused = 0.0;
  PB_GRID_STRIDE(i, n) {
    const float st = sqrtf(T.at((uint32_t)i));
    const float sv = (1.f * st) * s[i];
    s[i] = sv;
    p[i] = sv;
    temp3[i] = st * sv;
    acc += static_cast<double>(sv) * static_cast<double>(sv);
  }
  if (reduce_last(acc, unused, partials, &cg->ticket)) {
    const double norms = sqrt(acc);
    cg->norms = norms;
    cg->norms0 = norms;
    cg->gamma = norms * norms;
    cg->normp = norms;
    cg->xmax = cg->normx;
    if (norms < k_eps) cg->done = 1;      // flag = 1
  }
}

// CG step, after q <- K temp3: q = 1 sqrt(S) q (gemv_functor3), |q|; delta, alpha (:303-315)
__global__ void __launch_bounds__(kBlock) cg_forward_tail_kernel(size_t m, ScaleRef S, float* __restrict__ q,
                                                                 CgState* cg, double* partials, double shift,
                                                                 double k_eps, const CrossSum cross) {
  if (cg->done) return;
  double acc = 0.0, unused = 0.0;
  PB_GRID_STRIDE(i, m) {
    const float qv = (1.f * sqrtf(S.at((uint32_t)i))) * q[i];
    q[i] = qv;
    acc += static_cast<double>(qv) * static_cast<double>(qv);
  }
  if (reduce_last(acc, unused, partials, &cg->ticket, &cross)) {
    cg->normq = sqrt(acc);
    double delta = cg->normq * cg->normq + shift * cg->normp * cg->normp;
    if (delta <= 0.) cg->indefinite = 1;
    if (delta == 0.) delta = k_eps;
    cg->alpha = static_cast<float>(cg->gamma / delta);
    cg->neg_alpha = static_cast<float>(-cg->gamma / delta);
  }
}

// x += alpha p, r -= alpha q (:319-322), s = x (:326), |x| (:350); head of gemv('t', 1, r, -shift, s)
__global__ void __launch_bounds__(kBlock) cg_update_kernel(size_t n, size_t m, ScaleRef T, ScaleRef S,
                                                           float neg_shift, float* __restrict__ x,
                                                           const float* __restrict__ p, float* __restrict__ r,
                                                           const float* __restrict__ q, float* __restrict__ s,
                                                           float* __restrict__ temp3, CgState* cg,
                                                           double* partials) {
  if (cg->done) return;
  const float alpha = cg->alpha, neg_alpha = cg->neg_alpha;
  double acc = 0.0, unused = 0.0;
  const size_t len = n > m ? n : m;
  PB_GRID_STRIDE(i, len) {
    if (i < n) {
      const float xv = fmaf(alpha, p[i], x[i]);
      x[i] = xv;
      acc += static_cast<double>(xv) * static_cast<double>(xv);
      s[i] = (neg_shift / (1.f * sqrtf(T.at((uint32_t)i)))) * xv;
    }
    if (i < m) {
      const float rv = fmaf(neg_alpha, q[i], r[i]);
      r[i] = rv;
      temp3[i] = sqrtf(S.at((uint32_t)i)) * rv;
    }
  }
  if (reduce_last(acc, unused, partials, &cg->ticket)) cg->normx = sqrt(acc);
}

// tail of gemv('t'): s = 1 sqrt(T) s, |s|; beta, convergence verdict (:337-355)
__global__ void __launch_bounds__(kBlock) cg_adjoint_tail_kernel(size_t n, ScaleRef T, float* __restrict__ s,
                                                                 CgState* cg, double* partials, double tol) {
  if (cg->done) return;
  double acc = 0.0, unused = 0.0;
  PB_GRID_STRIDE(i, n) {
    const float sv = (1.f * sqrtf(T.at((uint32_t)i))) * s[i];
    s[i] = sv;
    acc += static_cast<double>(sv) * static_cast<double>(sv);
  }
  if (reduce_last(acc, unused, partials, &cg->ticket)) {
    const double norms = sqrt(acc);
    cg->norms = norms;
    const double gamma1 = cg->gamma;
    cg->gamma = norms * norms;
    cg->beta = static_cast<float>(cg->gamma / gamma1);
    cg->xmax = fmax(cg->xmax, cg->normx);
    const bool converged = (norms <= cg->norms0 * tol) || (cg->normx * tol >= 1.);
    // the reference still forms p = s + beta p before leaving the loop (:343-347); p is scratch
    // (x_half) that the prox overwrites, so the step can stop here
    if (converged) cg->done = 1;
    else cg->k = cg->k + 1;
  }
}

// p = s + beta p (:343-347), |p| (:300); head of the next gemv('n', 1, p, 0, q): temp3 = sqrt(T) p
__global__ void __launch_bounds__(kBlock) cg_direction_kernel(size_t n, ScaleRef T, float* __restrict__ s,
                                                              float* __restrict__ p,
                                                              float* __restrict__ temp3, CgState* cg,
                                                              double* partials) {
  if (cg->done) return;
  const float beta = cg->beta;
  double acc = 0.0, unused = 0.0;
  PB_GRID_STRIDE(i, n) {
    const float pv = fmaf(beta, p[i], s[i]);
    s[i] = pv;
    p[i] = pv;
    temp3[i] = sqrtf(T.at((uint32_t)i)) * pv;
    acc += static_cast<double>(pv) * static_cast<double>(pv);
  }
  if (reduce_last(acc, unused, partials, &cg->ticket)) cg->normp = sqrt(acc);
}

// ---- outer iteration, part 2 (backend_admm.cu:438-523) ------------------------------------------
// temp3 = x_proj (:439);  x_proj = sqrt(T) (x_proj + temp1)            x_proj_functor :93-103
__global__ void __launch_bounds__(kBlock) admm_xproj_kernel(size_t n, ScaleRef T, float* __restrict__ x_proj,
                                                            const float* __restrict__ temp1,
                                                            float* __restrict__ temp3) {
  PB_GRID_STRIDE(i, n) {
    const float xv = x_proj[i];
    temp3[i] = xv;
    x_proj[i] = sqrtf(T.at((uint32_t)i)) * (xv + temp1[i]);
  }
}

// x_dual = temp1 sqrt(T) - x_proj (:105-115); z_dual = temp2 / sqrt(S) - z_proj (:117-127);
// temp1 = x_proj - x_dual; temp2 = z_proj - z_dual (:81-91)
__global__ void __launch_bounds__(kBlock) admm_dual_kernel(size_t n, size_t m, ScaleRef T, ScaleRef S,
                                                           const float* __restrict__ x_proj,
                                                           float* __restrict__ x_dual,
                                                           const float* __restrict__ z_proj,
                                                           float* __restrict__ z_dual, float* __restrict__ temp1,
                                                           float* __restrict__ temp2) {
  const size_t len = n > m ? n : m;
  PB_GRID_STRIDE(i, len) {
    if (i < n) {
      const float xp = x_proj[i];
      const float xd = temp1[i] * sqrtf(T.at((uint32_t)i)) - xp;
      x_dual[i] = xd;
      temp1[i] = xp - xd;
    }
    if (i < m) {
      const float zp = z_proj[i];
      const float zd = temp2[i] / sqrtf(S.at((uint32_t)i)) - zp;
      z_dual[i] = zd;
      temp2[i] = zp - zd;
    }
  }
}

// ---- residuals (backend_admm.cu:529-626) --------------------------------------------------------
// sums[0] = |sqrt(S)(K x_half - z_half)|^2 (kxz holds K x_half - z_half), sums[1] = |sqrt(S) z_half|^2
__global__ void __launch_bounds__(kBlock) admm_primal_residual_kernel(size_t m, ScaleRef S,
                                                                      const float* __restrict__ kxz,
                                                                      const float* __restrict__ z_half,
                                                                      double* partials, unsigned* ticket,
                                                                      double* sums, const CrossSum cross) {
  double a = 0.0, b = 0.0;
  PB_GRID_STRIDE(i, m) {
    const float ss = sqrtf(S.at((uint32_t)i));
    const float v = ss * kxz[i];
    const float u = ss * z_half[i];
    a += static_cast<double>(v) * static_cast<double>(v);
    b += static_cast<double>(u) * static_cast<double>(u);
  }
  if (reduce_last(a, b, partials, ticket, &cross)) { sums[0] = a; sums[1] = b; }
}

// w = -rho T^-1 (x_half - x_proj + x_dual) -> temp1, sums[3] = |sqrt(T) w|^2;
// y = -rho S^1 (z_half - z_proj + z_dual) -> temp2                      get_dual_functor :184-196
__global__ void __launch_bounds__(kBlock) admm_dual_variables_kernel(
    size_t n, size_t m, float rho, ScaleRef T, ScaleRef S, const float* __restrict__ x_half,
    const float* __restrict__ x_proj, const float* __restrict__ x_dual, const float* __restrict__ z_half,
    const float* __restrict__ z_proj, const float* __restrict__ z_dual, float* __restrict__ w_out,
    float* __restrict__ y_out, double* partials, unsigned* ticket, double* sums) {
  double a = 0.0, unused = 0.0;
  const size_t len = n > m ? n : m;
  PB_GRID_STRIDE(i, len) {
    if (i < n && w_out) {
      const float t = T.at((uint32_t)i);
      const float w = -rho * powf(t, -1.f) * (x_half[i] - x_proj[i] + x_dual[i]);
      w_out[i] = w;
      const float sw = sqrtf(t) * w;
      a += static_cast<double>(sw) * static_cast<double>(sw);
    }
    if (i < m && y_out) {
      const float sg = S.at((uint32_t)i);
      y_out[i] = -rho * powf(sg, 1.f) * (z_half[i] - z_proj[i] + z_dual[i]);
    }
  }
  if (sums) {
    if (reduce_last(a, unused, partials, ticket)) sums[3] = a;
  }
}

// sums[2] = |sqrt(T)(w + K^T y)|^2
__global__ void __launch_bounds__(kBlock) admm_dual_residual_kernel(size_t n, ScaleRef T,
                                                                    const float* __restrict__ wkty,
                                                                    double* partials, unsigned* ticket,
                                                                    double* sums) {
  double a = 0.0, unused = 0.0;
  PB_GRID_STRIDE(i, n) {
    const float v = sqrtf(T.at((uint32_t)i)) * wkty[i];
    a += static_cast<double>(v) * static_cast<double>(v);
  }
  if (reduce_last(a, unused, partials, ticket)) sums[2] = a;
}

__global__ void __launch_bounds__(kBlock) admm_rescale_kernel(size_t n, size_t m, float f,
                                                              float* __restrict__ x_dual,
                                                              float* __restrict__ z_dual) {
  const size_t len = n > m ? n : m;
  PB_GRID_STRIDE(i, len) {
    if (i < n) x_dual[i] = f * x_dual[i];
    if (i < m) z_dual[i] = f * z_dual[i];
  }
}

__global__ void __launch_bounds__(kBlock) admm_scale_tail_kernel(float* __restrict__ v, size_t n, float beta,
                                                                 const int* __restrict__ skip) {
  if (skip && *skip) return;
  PB_GRID_STRIDE(i, n) v[i] = beta * v[i];
}

// row-sharded adjoint: res = beta res + (sum over ranks of the partial K^T rhs)
__global__ void __launch_bounds__(kBlock) admm_axpby_kernel(float* __restrict__ res, const float* __restrict__ part,
                                                            size_t n, float beta, const int* __restrict__ skip) {
  if (skip && *skip) return;
  PB_GRID_STRIDE(i, n) res[i] = beta == 0.f ? part[i] : beta * res[i] + part[i];
}

}  // namespace

class BackendADMM : public Backend {
 public:
  BackendADMM(Context* ctx, std::shared_ptr<Problem> prob, const pb_admm_options& opts,
              const pb_solver_options& sopts)
      : Backend(ctx, std::move(prob), sopts), opts_(opts) {}
  ~BackendADMM() override {
    if (ctx_->skip_flag == skip_done() || ctx_->skip_flag == skip_init()) ctx_->skip_flag = nullptr;
  }

  void initialize(const float* h_x0, size_t nx0, const float* h_y0, size_t ny0) override;
  void iterate(int n_iters) override;
  void profile(int n_iters, float out_ms[3]) override;
  void residuals(float out[6]) override;
  void stepsizes(double out[3]) override {
    out[0] = rho_;
    out[1] = delta_;
    out[2] = static_cast<double>(cg_steps_total());
  }
  size_t iteration() const override { return iteration_; }
  void current_solution(float* h_x, float* h_z, float* h_y, float* h_w) override;
  size_t gpu_mem_amount() const override {                 // backend_admm.cu:743-750
    const size_t m = problem_->nrows(), n = problem_->ncols();
    return (4 * (n + m) + std::max(m, n)) * sizeof(float);
  }
  void device_iterates(float** d_x, float** d_y) override {
    if (d_x) *d_x = x_half_.data();
    if (d_y) *d_y = nullptr;        // the dual iterate is implicit: y = -rho S (z_half - z_proj + z_dual)
  }
  int residual_iter() const override { return opts_.residual_iter; }
  // Row-sharded ADMM over the GPUs of one box (SURVEY.md 8(e)): this rank's Problem holds a block of ROWS of K and
  // of the f-side vectors; the n-side vectors are replicated.  K x is local; K^T r is summed over ranks with one
  // ncclAllReduce of n floats per adjoint apply; the sums over rows (|q|^2, primal residual) are combined inside
  // the reduction kernels (pb_crosssum.cuh); sums over columns are computed redundantly and identically.
  void set_slab(Comm* comm) override { comm_ = comm; }
  // residuals refresh AFTER iteration_++ (backend_admm.cu:525-529)
  bool refreshes_on(size_t it_before) const override {
    const unsigned long long mod = static_cast<unsigned long long>(static_cast<long long>(opts_.residual_iter));
    return ((it_before + 1) % mod) == 0;
  }

 private:
  unsigned egrid(size_t items) const {
    return static_cast<unsigned>(std::min<size_t>(grid_for(items), (size_t)ctx_->num_sms * 8));
  }
  const int* skip_done() const { return d_cg_.data() ? &d_cg_.data()->done : nullptr; }
  const int* skip_init() const { return d_cg_.data() ? &d_cg_.data()->skip_init : nullptr; }
  // result = beta * result + K rhs (or K^T rhs) on full-length vectors; rows / columns beyond the
  // operator's extent see K = 0 (linearoperator.cu:134-170 scales or fills the whole vector)
  void apply(float* d_res, const float* d_rhs, float beta, bool transpose, const int* skip);
  void project_onto_graph(double cg_tol);
  void update_residuals();
  long long cg_steps_total();

  pb_admm_options opts_;
  Comm* comm_ = nullptr;
  bool sharded() const { return comm_ && comm_->world() > 1; }
  CrossSum cross() const { return sharded() ? comm_->cross_sum() : CrossSum(); }
  unsigned long long global_rows_ = 0;
  DeviceBuffer<float> kt_part_;        // row-sharded: this rank's partial K^T rhs
  DeviceBuffer<float> x_half_, z_half_, x_proj_, z_proj_, x_dual_, z_dual_, temp1_, temp2_, temp3_;
  DeviceBuffer<CgState> d_cg_;
  DeviceBuffer<double> d_part_, d_sums_;
  DeviceBuffer<unsigned> d_ticket_;
  DeviceBuffer<long long> d_cg_total_;
  ProxList prox_g_, prox_f_;
  float rho_ = 1.f, delta_ = 1.f;
  int arb_u_ = 0, arb_l_ = 0;
  size_t iteration_ = 0;
  // the reference leaves these uninitialised until the first refresh (backend.hpp:82-92); FLT_MAX
  // keeps Solver::Solve from reporting convergence before residuals exist
  float primal_residual_ = std::numeric_limits<float>::max(), dual_residual_ = std::numeric_limits<float>::max();
  float primal_var_norm_ = 0.f, dual_var_norm_ = 0.f;
  cudaEvent_t* prof_ev_ = nullptr;
};

// counts CG steps on the device so tests can compare the step count with the reference's
__global__ void cg_count_kernel(const CgState* __restrict__ cg, long long* total) {
  if (threadIdx.x == 0 && blockIdx.x == 0) *total += cg->k;
}

long long BackendADMM::cg_steps_total() {
  long long v = 0;
  if (d_cg_total_.size()) {
    d_cg_total_.download(&v, 1, ctx_->stream);
    PB_CUDA(cudaStreamSynchronize(ctx_->stream));
  }
  return v;
}

void BackendADMM::initialize(const float*, size_t, const float*, size_t) {
  // BackendADMM::Initialize ignores Solver::Options::x0 / y0 (backend_admm.cu:285-352)
  ctx_->bind();
  if (!problem_->initialized()) fail(PB_ERR_INVALID, "Problem has not been initialized.");
  if (problem_->dualized())
    fail(PB_ERR_UNSUPPORTED, "BackendADMM: solve_dual_problem is not supported (the reference's "
                             "DualLinearOperator drops the sign of beta = 1 accumulations, "
                             "dual_linearoperator.cu:43-58, which ADMM relies on)");
  const size_t m = problem_->nrows(), n = problem_->ncols();
  if (std::max(m, n) >= (1ull << 31)) fail(PB_ERR_UNSUPPORTED, "BackendADMM: more than 2^31-1 variables");
  cudaStream_t s = ctx_->stream;
  global_rows_ = m;
  if (sharded()) {
    // every rank must come to the same verdict before anybody throws (the next call is collective)
    const bool alpha = problem_->scaling_type() == Problem::kScalingAlpha;
    double v[3] = {alpha ? 1.0 : 0.0, static_cast<double>(m), static_cast<double>(n)};
    comm_->allreduce_sum_host(v, 3);
    if (v[0] != 0.0 && v[0] != comm_->world())
      fail(PB_ERR_INVALID, "row-sharded ADMM: ranks disagree on the scaling type");
    if (v[2] != static_cast<double>(n) * comm_->world())
      fail(PB_ERR_INVALID, "row-sharded ADMM: ranks disagree on the number of columns");
    global_rows_ = static_cast<unsigned long long>(v[1]);
    // alpha scaling: the preconditioners of the whole operator replace the rank-local ones
    if (alpha) problem_->shard_alpha_scaling(*comm_);
    comm_->ensure_halo(4);             // maps every rank's control block (reduction slots)
    if (!comm_->reduce_p2p())
      fail(PB_ERR_UNSUPPORTED, "row-sharded ADMM needs peer-to-peer access between the GPUs (CUDA IPC)");
  }
  try {
    if (sharded()) kt_part_.resize(n);
    x_half_.resize(n); x_proj_.resize(n); x_dual_.resize(n);
    z_half_.resize(m); z_proj_.resize(m); z_dual_.resize(m);
    temp1_.resize(n); temp2_.resize(m); temp3_.resize(std::max(m, n));
    d_cg_.resize(1);
    d_part_.resize(2 * (size_t)ctx_->num_sms * 8);
    d_sums_.resize(4);
    d_ticket_.resize(1);
    d_cg_total_.resize(1);
  } catch (Error& e) {
    if (e.status == PB_ERR_OOM) fail(PB_ERR_OOM, std::string("Out of memory: ") + e.what());
    throw;
  }
  x_half_.zero(s); x_proj_.zero(s); x_dual_.zero(s); z_half_.zero(s); z_proj_.zero(s); z_dual_.zero(s);
  temp1_.zero(s); temp2_.zero(s); temp3_.zero(s);
  d_cg_.zero(s); d_sums_.zero(s); d_ticket_.zero(s); d_cg_total_.zero(s);

  prox_g_.clear();
  prox_f_.clear();
  if (problem_->prox_g().empty()) {                        // :313-327
    if (problem_->prox_gstar().empty()) fail(PB_ERR_INVALID, "Neither prox_g nor prox_gstar specified.");
    for (auto& p : problem_->prox_gstar()) prox_g_.push_back(make_prox_moreau(ctx_, p));
  } else {
    prox_g_ = problem_->prox_g();
  }
  if (problem_->prox_f().empty()) {                        // :329-343
    if (problem_->prox_fstar().empty()) fail(PB_ERR_INVALID, "Neither prox_f nor prox_fstar specified.");
    for (auto& p : problem_->prox_fstar()) prox_f_.push_back(make_prox_moreau(ctx_, p));
  } else {
    prox_f_ = problem_->prox_f();
  }
  delta_ = opts_.arb_delta;                                // :345-348
  rho_ = static_cast<float>(opts_.rho0);
  iteration_ = 0;
  arb_u_ = arb_l_ = 0;
  primal_residual_ = dual_residual_ = std::numeric_limits<float>::max();
  primal_var_norm_ = dual_var_norm_ = 0.f;
  PB_CUDA(cudaStreamSynchronize(s));
}

void BackendADMM::apply(float* d_res, const float* d_rhs, float beta, bool transpose, const int* skip) {
  LinearOperator* K = problem_->linop();
  ctx_->skip_flag = skip;
  if (transpose && sharded()) {
    // partial K^T rhs of this rank's rows -> sum over ranks -> res = beta res + sum.  The all-reduce is a host-
    // enqueued collective and runs even when the device-side skip flag is set (its result is then not used).
    const size_t n = problem_->ncols();
    K->eval(kt_part_.data(), d_rhs, 0.f, true);
    if (n > K->ncols()) PB_CUDA(cudaMemsetAsync(kt_part_.data() + K->ncols(), 0, (n - K->ncols()) * sizeof(float), ctx_->stream));
    comm_->allreduce_sum_f32(kt_part_.data(), n);
    admm_axpby_kernel<<<egrid(n), kBlock, 0, ctx_->stream>>>(d_res, kt_part_.data(), n, beta, skip);
    PB_CHECK_LAUNCH();
    ctx_->launches++;
    ctx_->skip_flag = nullptr;
    return;
  }
  K->eval(d_res, d_rhs, beta, transpose);
  const size_t covered = transpose ? K->ncols() : K->nrows();
  const size_t total = transpose ? problem_->ncols() : problem_->nrows();
  if (total > covered) {
    if (beta == 0.f) {
      PB_CUDA(cudaMemsetAsync(d_res + covered, 0, (total - covered) * sizeof(float), ctx_->stream));
    } else if (beta != 1.f) {
      admm_scale_tail_kernel<<<egrid(total - covered), kBlock, 0, ctx_->stream>>>(d_res + covered, total - covered,
                                                                                  beta, skip);
      PB_CHECK_LAUNCH();
      ctx_->launches++;
    }
  }
  ctx_->skip_flag = nullptr;
}

// Minimise |K~ x - d|^2 + |x|^2 with CGLS on K~ = S^{1/2} K T^{1/2} (backend_admm.cu:385-436,
// cgls.hpp:222-371).  Vector aliases as in the reference: p = x_half, q = z_half, r = z_proj,
// s = x_dual, b = z_dual, x = x_proj.
void BackendADMM::project_onto_graph(double cg_tol) {
  const size_t m = problem_->nrows(), n = problem_->ncols();
  const size_t len = std::max(m, n);
  cudaStream_t st = ctx_->stream;
  const ScaleRef T = problem_->right_ref(), S = problem_->left_ref();
  CgState* cg = d_cg_.data();
  double* part = d_part_.data();
  const double shift = 1.0;
  const float neg_shift = static_cast<float>(-shift);
  const double k_eps = std::numeric_limits<float>::epsilon();
  float* x = x_proj_.data();
  float* p = x_half_.data();
  float* q = z_half_.data();
  float* r = z_proj_.data();
  float* s = x_dual_.data();
  float* b = z_dual_.data();

  admm_begin_kernel<<<egrid(len), kBlock, 0, st>>>(n, m, static_cast<float>(opts_.alpha), T, S, x_half_.data(), x,
                                                   s, z_half_.data(), b, temp1_.data(), temp2_.data(),
                                                   temp3_.data(), cg, part);
  PB_CHECK_LAUNCH();
  apply(b, temp3_.data(), 1.f, false, nullptr);                      // b += K (T^{1/2} temp1)
  admm_rhs_kernel<<<egrid(len), kBlock, 0, st>>>(n, m, T, S, x, b, r, temp3_.data(), cg);
  PB_CHECK_LAUNCH();
  apply(r, temp3_.data(), 1.f, false, skip_init());                  // r = b - K~ x   (if |x| > 0)
  cg_adjoint_head_kernel<<<egrid(len), kBlock, 0, st>>>(n, m, T, S, neg_shift, r, s, temp3_.data(), cg);
  PB_CHECK_LAUNCH();
  apply(s, temp3_.data(), 1.f, true, nullptr);                       // s = K~^T r - shift x
  cg_init_tail_kernel<<<egrid(n), kBlock, 0, st>>>(n, T, s, p, temp3_.data(), cg, part, k_eps);
  PB_CHECK_LAUNCH();
  ctx_->launches += 4;

  for (int k = 0; k < opts_.cg_max_iter; ++k) {
    apply(q, temp3_.data(), 0.f, false, skip_done());                // q = K~ p
    cg_forward_tail_kernel<<<egrid(m), kBlock, 0, st>>>(m, S, q, cg, part, shift, k_eps, cross());
    PB_CHECK_LAUNCH();
    cg_update_kernel<<<egrid(len), kBlock, 0, st>>>(n, m, T, S, neg_shift, x, p, r, q, s, temp3_.data(), cg, part);
    PB_CHECK_LAUNCH();
    apply(s, temp3_.data(), 1.f, true, skip_done());                 // s = K~^T r - shift x
    cg_adjoint_tail_kernel<<<egrid(n), kBlock, 0, st>>>(n, T, s, cg, part, cg_tol);
    PB_CHECK_LAUNCH();
    cg_direction_kernel<<<egrid(n), kBlock, 0, st>>>(n, T, s, p, temp3_.data(), cg, part);
    PB_CHECK_LAUNCH();
    ctx_->launches += 4;
  }
  cg_count_kernel<<<1, 32, 0, st>>>(cg, d_cg_total_.data());
  PB_CHECK_LAUNCH();
  ctx_->launches++;
}

void BackendADMM::update_residuals() {                     // backend_admm.cu:529-660
  const size_t m = problem_->nrows(), n = problem_->ncols();
  const size_t len = std::max(m, n);
  cudaStream_t st = ctx_->stream;
  const ScaleRef T = problem_->right_ref(), S = problem_->left_ref();
  double* part = d_part_.data();
  unsigned* ticket = d_ticket_.data();

  PB_CUDA(cudaMemcpyAsync(temp2_.data(), z_half_.data(), m * sizeof(float), cudaMemcpyDeviceToDevice, st));
  apply(temp2_.data(), x_half_.data(), -1.f, false, nullptr);        // K x_half - z_half
  admm_primal_residual_kernel<<<egrid(m), kBlock, 0, st>>>(m, S, temp2_.data(), z_half_.data(), part, ticket,
                                                           d_sums_.data(), cross());
  PB_CHECK_LAUNCH();
  admm_dual_variables_kernel<<<egrid(len), kBlock, 0, st>>>(n, m, rho_, T, S, x_half_.data(), x_proj_.data(),
                                                            x_dual_.data(), z_half_.data(), z_proj_.data(),
                                                            z_dual_.data(), temp1_.data(), temp2_.data(), part,
                                                            ticket, d_sums_.data());
  PB_CHECK_LAUNCH();
  apply(temp1_.data(), temp2_.data(), 1.f, true, nullptr);           // w + K^T y
  admm_dual_residual_kernel<<<egrid(n), kBlock, 0, st>>>(n, T, temp1_.data(), part, ticket, d_sums_.data());
  PB_CHECK_LAUNCH();
  ctx_->launches += 3;
  double sums[4];
  d_sums_.download(sums, 4, st);
  PB_CUDA(cudaStreamSynchronize(st));
  // cublasSnrm2 returns float (backend_admm.cu:46-50)
  primal_residual_ = static_cast<float>(std::sqrt(sums[0]));
  primal_var_norm_ = static_cast<float>(std::sqrt(sums[1]));
  dual_residual_ = static_cast<float>(std::sqrt(sums[2]));
  dual_var_norm_ = static_cast<float>(std::sqrt(sums[3]));

  const float eps_p = pdhg_eps(global_rows_, sopts_.tol_abs_primal, sopts_.tol_rel_primal, primal_var_norm_);
  const float eps_d = pdhg_eps(n, sopts_.tol_abs_dual, sopts_.tol_rel_dual, dual_var_norm_);
  const float rho_prev = rho_;
  const float t_it = opts_.arb_tau * static_cast<float>(iteration_);
  if ((dual_residual_ < eps_d) && (t_it > static_cast<float>(arb_l_))) {         // :629-634
    rho_ *= delta_;
    delta_ *= opts_.arb_gamma;
    arb_u_ = static_cast<int>(iteration_);
  } else if ((primal_residual_ < eps_p) && (t_it > static_cast<float>(arb_u_))) { // :635-640
    rho_ /= delta_;
    delta_ *= opts_.arb_gamma;
    arb_l_ = static_cast<int>(iteration_);
  }
  if (std::abs(rho_ - rho_prev) > 1e-7) {                  // :643-659
    admm_rescale_kernel<<<egrid(len), kBlock, 0, st>>>(n, m, rho_prev / rho_, x_dual_.data(), z_dual_.data());
    PB_CHECK_LAUNCH();
    ctx_->launches++;
  }
}

void BackendADMM::iterate(int n_iters) {
  ctx_->bind();
  const size_t m = problem_->nrows(), n = problem_->ncols();
  const size_t len = std::max(m, n);
  cudaStream_t st = ctx_->stream;
  const ScaleRef T = problem_->right_ref(), S = problem_->left_ref();
  for (int it = 0; it < n_iters; ++it) {
    if (prof_ev_) PB_CUDA(cudaEventRecord(prof_ev_[0], st));
    double cg_tol = opts_.cg_tol_min / std::pow(static_cast<float>(iteration_ + 1), opts_.cg_tol_pow);   // :403-405
    cg_tol = std::max(cg_tol, opts_.cg_tol_max);
    project_onto_graph(cg_tol);
    if (prof_ev_) PB_CUDA(cudaEventRecord(prof_ev_[1], st));

    admm_xproj_kernel<<<egrid(n), kBlock, 0, st>>>(n, T, x_proj_.data(), temp1_.data(), temp3_.data());
    PB_CHECK_LAUNCH();
    apply(z_proj_.data(), x_proj_.data(), 0.f, false, nullptr);      // z_proj = K x_proj (:456)
    admm_dual_kernel<<<egrid(len), kBlock, 0, st>>>(n, m, T, S, x_proj_.data(), x_dual_.data(), z_proj_.data(),
                                                    z_dual_.data(), temp1_.data(), temp2_.data());
    PB_CHECK_LAUNCH();
    ctx_->launches += 2;
    for (auto& p : prox_g_) p->eval(x_half_.data(), temp1_.data(), problem_->scaling_right(), 1 / rho_, false);
    for (auto& p : prox_f_) p->eval(z_half_.data(), temp2_.data(), problem_->scaling_left(), rho_, true);
    iteration_++;
    if (prof_ev_) PB_CUDA(cudaEventRecord(prof_ev_[2], st));

    const unsigned long long mod = static_cast<unsigned long long>(static_cast<long long>(opts_.residual_iter));
    if (iteration_ == 0 || (iteration_ % mod) == 0) update_residuals();
    if (prof_ev_) PB_CUDA(cudaEventRecord(prof_ev_[3], st));
  }
}

// average device ms per outer iteration of { CGLS projection, prox + dual updates, residuals }
void BackendADMM::profile(int n_iters, float out_ms[3]) {
  ctx_->bind();
  out_ms[0] = out_ms[1] = out_ms[2] = 0.f;
  cudaEvent_t ev[4];
  for (auto& e : ev) PB_CUDA(cudaEventCreate(&e));
  double acc[3] = {0, 0, 0};
  for (int i = 0; i < n_iters; ++i) {
    prof_ev_ = ev;
    iterate(1);
    prof_ev_ = nullptr;
    PB_CUDA(cudaEventSynchronize(ev[3]));
    for (int k = 0; k < 3; ++k) {
      float ms = 0.f;
      PB_CUDA(cudaEventElapsedTime(&ms, ev[k], ev[k + 1]));
      acc[k] += ms;
    }
  }
  for (auto& e : ev) cudaEventDestroy(e);
  if (n_iters > 0)
    for (int k = 0; k < 3; ++k) out_ms[k] = static_cast<float>(acc[k] / n_iters);
}

void BackendADMM::residuals(float out[6]) {
  ctx_->bind();
  PB_CUDA(cudaStreamSynchronize(ctx_->stream));
  out[0] = primal_residual_;
  out[1] = dual_residual_;
  out[2] = primal_var_norm_;
  out[3] = dual_var_norm_;
  out[4] = pdhg_eps(sharded() ? global_rows_ : problem_->nrows(), sopts_.tol_abs_primal, sopts_.tol_rel_primal,
                    primal_var_norm_);
  out[5] = pdhg_eps(problem_->ncols(), sopts_.tol_abs_dual, sopts_.tol_rel_dual, dual_var_norm_);
}

void BackendADMM::current_solution(float* h_x, float* h_z, float* h_y, float* h_w) {   // :697-741
  ctx_->bind();
  const size_t m = problem_->nrows(), n = problem_->ncols();
  const size_t len = std::max(m, n);
  cudaStream_t st = ctx_->stream;
  if (h_w || h_y) {
    admm_dual_variables_kernel<<<egrid(len), kBlock, 0, st>>>(
        n, m, rho_, problem_->right_ref(), problem_->left_ref(), x_half_.data(), x_proj_.data(), x_dual_.data(),
        z_half_.data(), z_proj_.data(), z_dual_.data(), h_w ? temp1_.data() : nullptr,
        h_y ? temp2_.data() : nullptr, nullptr, nullptr, nullptr);
    PB_CHECK_LAUNCH();
    ctx_->launches++;
  }
  if (h_w) download_to_host(ctx_, h_w, temp1_.data(), n);
  if (h_y) download_to_host(ctx_, h_y, temp2_.data(), m);
  if (h_x) download_to_host(ctx_, h_x, x_half_.data(), n);
  if (h_z) download_to_host(ctx_, h_z, z_half_.data(), m);
  PB_CUDA(cudaStreamSynchronize(st));
}

std::shared_ptr<Backend> make_backend_admm(Context* ctx, std::shared_ptr<Problem> prob,
                                           const pb_admm_options& opts, const pb_solver_options& sopts) {
  return std::make_shared<BackendADMM>(ctx, std::move(prob), opts, sopts);
}

}  // namespace pb
