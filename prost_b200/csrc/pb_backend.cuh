// pb_backend.cuh -- Backend base (include/prost/backend/backend.hpp:37-95) and the PDHG
// step-size state machine shared by host (unfused path) and device (fused path).
#pragma once

#include <cmath>
#include <memory>

#include "pb_problem.cuh"

namespace pb {

// Scalar state of BackendPDHG (backend_pdhg.hpp:132-156).  In fused mode it lives in device
// memory and is advanced by a one-CTA kernel, so iterations need no host round trip.
struct PdhgState {
  float tau, sigma, theta;
  float arg_alpha;
  int arb_l, arb_u;
  unsigned long long iteration;     // iteration_ (incremented after the residual block)
  // refreshed on residual iterations only (backend_pdhg.cu:433-436)
  float primal_residual, dual_residual, primal_var_norm, dual_var_norm;
  float eps_primal, eps_dual;
};

struct PdhgParams {
  int stepsize_variant;
  float alg2_gamma, arg_nu, arg_delta, arb_delta, arb_tau;
  float tol_rel_primal, tol_rel_dual, tol_abs_primal, tol_abs_dual;
  unsigned long long nrows, ncols;
};

// eps_primal / eps_dual (backend.hpp:71-74): sqrt(size_t) is double, times float tolerance,
// plus the float product tol_rel * norm, returned as float.
__host__ __device__ inline float pdhg_eps(unsigned long long n, float tol_abs, float tol_rel,
                                          float var_norm) {
  return static_cast<float>(sqrt(static_cast<double>(n)) * static_cast<double>(tol_abs) +
                            static_cast<double>(tol_rel * var_norm));
}

// UpdateResidualsAndStepsizes after the four sums are known (backend_pdhg.cu:433-488).
// sums = { sum diff_p^2, sum z_hat^2, sum diff_d^2, sum w_hat^2 }; `check` says whether this
// iteration refreshed them.  Also performs iteration_++ (:374).
__host__ __device__ inline void pdhg_update(PdhgState& s, const PdhgParams& p, const double* sums,
                                            bool check) {
  if (check) {
    s.primal_residual = sqrtf(static_cast<float>(sums[0]));
    s.primal_var_norm = sqrtf(static_cast<float>(sums[1]));
    s.dual_residual = sqrtf(static_cast<float>(sums[2]));
    s.dual_var_norm = sqrtf(static_cast<float>(sums[3]));
    const float eps_p = pdhg_eps(p.nrows, p.tol_abs_primal, p.tol_rel_primal, s.primal_var_norm);
    const float eps_d = pdhg_eps(p.ncols, p.tol_abs_dual, p.tol_rel_dual, s.dual_var_norm);
    s.eps_primal = eps_p;
    s.eps_dual = eps_d;
    if (p.stepsize_variant == PB_PDHG_GOLDSTEIN) {            // :443-460
      const float scale = eps_d / eps_p;
      if (s.dual_residual > scale * s.primal_residual * p.arg_delta) {
        s.tau = s.tau / (1 - s.arg_alpha);
        s.sigma = s.sigma * (1 - s.arg_alpha);
        s.arg_alpha = s.arg_alpha * p.arg_nu;
      }
      if (s.dual_residual < scale * s.primal_residual / p.arg_delta) {
        s.tau = s.tau * (1 - s.arg_alpha);
        s.sigma = s.sigma / (1 - s.arg_alpha);
        s.arg_alpha = s.arg_alpha * p.arg_nu;
      }
    } else if (p.stepsize_variant == PB_PDHG_BOYD) {          // :462-476
      const float t_it = p.arb_tau * static_cast<float>(s.iteration);
      if (s.dual_residual < eps_d && t_it > static_cast<float>(s.arb_l)) {
        s.tau /= p.arb_delta;
        s.sigma *= p.arb_delta;
        s.arb_u = static_cast<int>(s.iteration);
      } else if (s.primal_residual < eps_p && t_it > static_cast<float>(s.arb_u)) {
        s.tau *= p.arb_delta;
        s.sigma /= p.arb_delta;
        s.arb_l = static_cast<int>(s.iteration);
      }
    }
  }
  if (p.stepsize_variant == PB_PDHG_ALG2) {                   // :483-488, double literals
    s.theta = static_cast<float>(
        1.0 / sqrt(1.0 + 2.0 * static_cast<double>(p.alg2_gamma) * static_cast<double>(s.tau)));
    s.tau = s.theta * s.tau;
    s.sigma = s.sigma / s.theta;
  }
  s.iteration++;
}

class Backend {
 public:
  Backend(Context* ctx, std::shared_ptr<Problem> prob, const pb_solver_options& sopts)
      : ctx_(ctx), problem_(std::move(prob)), sopts_(sopts) {}
  virtual ~Backend() {}

  virtual void initialize(const float* h_x0, size_t nx0, const float* h_y0, size_t ny0) = 0;
  virtual void iterate(int n_iters) = 0;
  virtual void profile(int n_iters, float out_ms[3]) { iterate(n_iters); out_ms[0] = out_ms[1] = out_ms[2] = 0.f; }
  virtual void profile_detail(int n_iters, float out[8]) {
    profile(n_iters, out);
    out[3] = 0.f; out[4] = static_cast<float>(n_iters); out[5] = out[6] = out[7] = 0.f;
  }
  // primal_residual, dual_residual, primal_var_norm, dual_var_norm, eps_primal, eps_dual
  virtual void residuals(float out[6]) = 0;
  virtual void stepsizes(double out[3]) = 0;
  virtual size_t iteration() const = 0;
  virtual void current_solution(float* h_x, float* h_z, float* h_y, float* h_w) = 0;
  virtual size_t gpu_mem_amount() const = 0;
  virtual bool is_fused() const { return false; }
  virtual unsigned long long one_pass_iterations() const { return 0; }
  virtual void device_iterates(float** d_x, float** d_y) = 0;
  // iterations between two residual refreshes
  virtual int residual_iter() const = 0;
  // does the iteration that starts with iteration() == it_before refresh the residuals?  PDHG checks
  // before iteration_++ (backend_pdhg.cu:389, size_t % int), ADMM after it (backend_admm.cu:525-529).
  virtual bool refreshes_on(size_t it_before) const {
    const unsigned long long mod = static_cast<unsigned long long>(static_cast<long long>(residual_iter()));
    return it_before == 0 || (it_before % mod) == 0;
  }
  // slab decomposition (pb_comm.cuh); must be called before initialize()
  virtual void set_slab(class Comm*) { fail(PB_ERR_UNSUPPORTED, "this backend has no slab decomposition"); }

  Context* ctx() const { return ctx_; }
  Problem* problem() const { return problem_.get(); }
  const pb_solver_options& solver_options() const { return sopts_; }
  // Solver::Initialize pushes its options into the backend (solver.cu:88-90); takes effect at initialize()
  void set_solver_options(const pb_solver_options& o) { sopts_ = o; }
  unsigned long long launch_base = 0;

 protected:
  Context* ctx_;
  std::shared_ptr<Problem> problem_;
  pb_solver_options sopts_;
};

std::shared_ptr<Backend> make_backend_pdhg(Context* ctx, std::shared_ptr<Problem> prob,
                                           const pb_pdhg_options& opts, const pb_solver_options& sopts);
std::shared_ptr<Backend> make_backend_admm(Context* ctx, std::shared_ptr<Problem> prob,
                                           const pb_admm_options& opts, const pb_solver_options& sopts);

}  // namespace pb
