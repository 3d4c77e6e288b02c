// pb_pdhg.cu -- BackendPDHG: the primal-dual hybrid gradient iteration.
// Reference: src/backend/backend_pdhg.cu (Initialize :199-309, PerformIteration :311-381,
// UpdateResidualsAndStepsizes :383-489, current_solution :513-563).
//
// Two execution modes with identical semantics:
//  * fused   -- two passes per iteration (pb_fused.cuh), 4 state vectors, step sizes and residual
//               bookkeeping in device memory, no host synchronisation inside iterate();
//  * unfused -- the reference's kernel sequence over 9 state vectors, used when the planner
//               cannot fuse (sparse/dense blocks, permuted or oversized prox groups, dualised
//               problems) and as an A/B check of the fused passes.
#include <algorithm>
#include <cmath>
#include <iostream>

#include "pb_backend.cuh"
#include "pb_comm.cuh"
#include "pb_fused.cuh"
#include "pb_reduce.cuh"
#include "pb_stencil.cuh"

namespace pb {

// ---- unfused kernels ----------------------------------------------------------------------------

// temp = x - tau * T * kty          (primal_proxarg_functor, backend_pdhg.cu:38-51)
__global__ void __launch_bounds__(kBlock) primal_proxarg_kernel(float* __restrict__ temp,
                                                                const float* __restrict__ x,
                                                                const float* __restrict__ T,
                                                                const float* __restrict__ kty, size_t n,
                                                                float tau) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x)
    temp[i] = primal_prox_arg(x[i], tau, T[i], kty[i]);
}

// temp = y + sigma * S * ((1+theta) kx - theta kx_prev)   (dual_proxarg_functor, :54-70)
__global__ void __launch_bounds__(kBlock) dual_proxarg_kernel(float* __restrict__ temp,
                                                              const float* __restrict__ y,
                                                              const float* __restrict__ S,
                                                              const float* __restrict__ kx,
                                                              const float* __restrict__ kx_prev, size_t m,
                                                              float sigma, float theta) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < m;
       i += (size_t)gridDim.x * blockDim.x)
    temp[i] = dual_prox_arg(y[i], sigma, S[i], dual_extrapolate(theta, kx[i], kx_prev[i]));
}

// primal_residual_transform (:97-120): per-CTA partial (sum diff^2, sum z_hat^2)
__global__ void __launch_bounds__(kBlock) primal_residual_kernel(
    const float* __restrict__ y_prev, const float* __restrict__ y, const float* __restrict__ S,
    const float* __restrict__ kx_prev, const float* __restrict__ kx, size_t m, float sigma, float theta,
    double* __restrict__ part) {
  double a = 0.0, b = 0.0;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < m;
       i += (size_t)gridDim.x * blockDim.x) {
    const float sq = sqrtf(S[i]);
    const float z_hat = (y_prev[i] - y[i]) / (sigma * sq) + sq * ((1 + theta) * kx[i] - theta * kx_prev[i]);
    const float diff = z_hat - sq * kx[i];
    a += static_cast<double>(diff * diff);
    b += static_cast<double>(z_hat * z_hat);
  }
  block_sum2(a, b);
  if (threadIdx.x == 0) { part[2 * blockIdx.x] = a; part[2 * blockIdx.x + 1] = b; }
}

// dual_residual_transform (:73-94)
__global__ void __launch_bounds__(kBlock) dual_residual_kernel(
    const float* __restrict__ x_prev, const float* __restrict__ x, const float* __restrict__ T,
    const float* __restrict__ kty_prev, const float* __restrict__ kty, size_t n, float tau,
    double* __restrict__ part) {
  double a = 0.0, b = 0.0;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x) {
    const float sq = sqrtf(T[i]);
    const float w_hat = (x_prev[i] - x[i]) / (tau * sq) - sq * kty_prev[i];
    const float diff = w_hat + sq * kty[i];
    a += static_cast<double>(diff * diff);
    b += static_cast<double>(w_hat * w_hat);
  }
  block_sum2(a, b);
  if (threadIdx.x == 0) { part[2 * blockIdx.x] = a; part[2 * blockIdx.x + 1] = b; }
}

// folds the primal and the dual partials into sums[0..3] (one CTA, index order)
__global__ void __launch_bounds__(kBlock) fold_residuals_kernel(const double* __restrict__ part_p,
                                                                unsigned np,
                                                                const double* __restrict__ part_d,
                                                                unsigned nd, double* __restrict__ sums) {
  double a, b;
  fold_partials2(part_p, np, a, b);
  if (threadIdx.x == 0) { sums[0] = a; sums[1] = b; }
  fold_partials2(part_d, nd, a, b);
  if (threadIdx.x == 0) { sums[2] = a; sums[3] = b; }
}

// fused mode: fold + step-size state machine on the device (one CTA)
__global__ void __launch_bounds__(kBlock) pdhg_finalize_kernel(PdhgState* __restrict__ st, PdhgParams prm,
                                                               const double* __restrict__ part_p,
                                                               unsigned np,
                                                               const double* __restrict__ part_d,
                                                               unsigned nd, unsigned long long iteration,
                                                               int check) {
  __shared__ double sums[4];
  if (check) {
    double a, b;
    fold_partials2(part_p, np, a, b);
    if (threadIdx.x == 0) { sums[0] = a; sums[1] = b; }
    fold_partials2(part_d, nd, a, b);
    if (threadIdx.x == 0) { sums[2] = a; sums[3] = b; }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    PdhgState s = *st;
    s.iteration = iteration;
    pdhg_update(s, prm, sums, check != 0);
    *st = s;
  }
}

// slab mode: the four sums were folded per rank and all-reduced; advance the state from them
__global__ void pdhg_finalize_sums_kernel(PdhgState* __restrict__ st, PdhgParams prm,
                                          const double* __restrict__ sums, unsigned long long iteration,
                                          int check) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    PdhgState s = *st;
    s.iteration = iteration;
    pdhg_update(s, prm, sums, check != 0);
    *st = s;
  }
}

// slab mode, current_solution only: K u and K^T p over the local columns with the neighbours' halo
// columns (same device functions, hence the same arithmetic, as the fused passes)
template <bool THREE_D>
__global__ void __launch_bounds__(kStencilBlock) slab_forward_kernel(const GradGeom g,
                                                                    const float* __restrict__ u,
                                                                    const float* __restrict__ u_halo,
                                                                    float* __restrict__ kx) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= g.plane) return;
  uint32_t xl, y, l, x;
  g.div_q.divmod(t, xl, y);            // q = ny (VEC = 1)
  g.div_nx.divmod(xl, l, x);
  const uint32_t idx = y + x * g.ny + l * g.nxny;
  float gx[1], gy[1], gl[1];
  grad_fwd<1, THREE_D, true>(g, u, u_halo, idx, x, y, l, gx, gy, gl);
  kx[idx] = gx[0];
  kx[g.plane + idx] = gy[0];
  if (THREE_D) kx[2u * (size_t)g.plane + idx] = gl[0];
  if (g.has_id) kx[g.id_row + idx] = __fmul_rn(u[idx], g.id_factor);
}

template <bool THREE_D, bool HAS_ID>
__global__ void __launch_bounds__(kStencilBlock) slab_adjoint_kernel(const GradGeom g,
                                                                    const float* __restrict__ p,
                                                                    const float* __restrict__ p_halo,
                                                                    float* __restrict__ kty) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= g.plane) return;
  uint32_t xl, y, l, x;
  g.div_q.divmod(t, xl, y);
  g.div_nx.divmod(xl, l, x);
  const uint32_t idx = y + x * g.ny + l * g.nxny;
  float out[1];
  grad_adj<1, THREE_D, HAS_ID, true>(g, p, p_halo, idx, x, y, l, out);
  kty[idx] = out[0];
}

// w = (x_prev - x) / (T tau) - kty_prev     (compute_w_variable_functor, :146-160)
__global__ void __launch_bounds__(kBlock) w_variable_kernel(float* __restrict__ w,
                                                            const float* __restrict__ x_prev,
                                                            const float* __restrict__ x,
                                                            const ScaleRef T,
                                                            const float* __restrict__ kty_prev, size_t n,
                                                            float tau) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x)
    w[i] = (x_prev[i] - x[i]) / ((T.ptr ? T.ptr[i] : T.val) * tau) - kty_prev[i];
}

// z = (y_prev - y) / (sigma S) + (1+theta) kx - theta kx_prev   (compute_z_variable_functor, :170-186)
__global__ void __launch_bounds__(kBlock) z_variable_kernel(float* __restrict__ z,
                                                            const float* __restrict__ y_prev,
                                                            const float* __restrict__ y,
                                                            const ScaleRef S,
                                                            const float* __restrict__ kx,
                                                            const float* __restrict__ kx_prev, size_t m,
                                                            float sigma, float theta) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < m;
       i += (size_t)gridDim.x * blockDim.x)
    z[i] = (y_prev[i] - y[i]) / (sigma * (S.ptr ? S.ptr[i] : S.val)) + (1 + theta) * kx[i] - theta * kx_prev[i];
}

// ---- backend -------------------------------------------------------------------------------------

class BackendPDHG : public Backend {
 public:
  BackendPDHG(Context* ctx, std::shared_ptr<Problem> prob, const pb_pdhg_options& opts,
              const pb_solver_options& sopts)
      : Backend(ctx, std::move(prob), sopts), opts_(opts) {
    if (opts_.residual_iter == 0) fail(PB_ERR_INVALID, "residual_iter must not be 0");
    if (opts_.stepsize_variant < PB_PDHG_ALG1 || opts_.stepsize_variant > PB_PDHG_BOYD)
      fail(PB_ERR_INVALID, "unknown PDHG step size variant");
  }

  void initialize(const float* h_x0, size_t nx0, const float* h_y0, size_t ny0) override;
  void iterate(int n_iters) override;
  void profile(int n_iters, float out_ms[3]) override;
  void profile_detail(int n_iters, float out[8]) override;
  void residuals(float out[6]) override;
  void stepsizes(double out[3]) override;
  size_t iteration() const override { return iteration_; }
  void current_solution(float* h_x, float* h_z, float* h_y, float* h_w) override;
  size_t gpu_mem_amount() const override {
    const size_t m = problem_->nrows(), n = problem_->ncols();
    if (fused_) return (2 * (n + m) + (tile_ok_ ? m : 0)) * sizeof(float);
    return (4 * (n + m) + std::max(n, m)) * sizeof(float);     // backend_pdhg.cu:503-511
  }
  bool is_fused() const override { return fused_; }
  unsigned long long one_pass_iterations() const override { return tile_iterations_; }
  void device_iterates(float** d_x, float** d_y) override { *d_x = x_.data(); *d_y = y_.data(); }
  int residual_iter() const override { return opts_.residual_iter; }
  void set_slab(Comm* comm) override { comm_ = comm; }

 private:
  // slab mode (comm_ != nullptr): slab-aware K / K^T
  DeviceBuffer<unsigned> fin_ticket_;        // RingFinish: CTAs of the running residual-refresh launch that are done
  RingFinish ring_finish();
  void slab_apply(float* d_res, const float* d_rhs, const float* d_halo, bool adjoint);
  Comm* comm_ = nullptr;
  bool is_check_iteration() const {
    // size_t % int of the reference: a negative residual_iter wraps to a huge modulus, i.e.
    // "only at iteration 0" (Appendix B #4)
    const unsigned long long mod = static_cast<unsigned long long>(static_cast<long long>(opts_.residual_iter));
    return iteration_ == 0 || (iteration_ % mod) == 0;
  }
  bool plan_fused();
  void iteration_fused();
  cudaEvent_t* prof_ev_ = nullptr;     // 4 events when profiling, else null
  void iteration_unfused();
  PdhgState fetch_state();
  unsigned sgrid(size_t n) const { return (unsigned)std::min<size_t>(grid_for(n), (size_t)ctx_->num_sms * 32); }

  pb_pdhg_options opts_;
  PdhgParams params_;
  ProxList prox_g_, prox_fstar_;
  bool fused_ = false;
  bool tile_ok_ = false;               // non-check iterations run as one tiled pass (pb_tile.cu)
  unsigned long long tile_iterations_ = 0, tile_check_iterations_ = 0;
  unsigned long long iteration_ = 0;

  // iterates: x_/y_ current, x_prev_/y_prev_ previous (ping-pong in fused mode)
  DeviceBuffer<float> x_, x_prev_, y_, y_prev_;
  // third dual buffer for tiled residual-refresh iterations (they read y^k AND y^{k-1} while writing y^{k+1})
  DeviceBuffer<float> y_stage_;
  float* y_prev_staging() {
    if (y_stage_.size() != y_.size()) y_stage_.resize(y_.size());
    return y_stage_.data();
  }
  // unfused only
  DeviceBuffer<float> temp_, kx_, kx_prev_, kty_, kty_prev_;
  // fused plan
  StencilPlan stencil_;                // specialised gradient passes where the structure matches
  BlockList blocks_;
  std::vector<ProxDesc> g_descs_, f_descs_;
  std::vector<ScaleRef> g_scale_, f_scale_;     // T / Sigma as seen by each prox (scalar when constant on its range)
  unsigned part_p_cap_ = 0, part_d_cap_ = 0;
  // state + reductions
  PdhgState h_state_;                  // master copy in unfused mode
  DeviceBuffer<PdhgState> d_state_;    // master copy in fused mode
  DeviceBuffer<double> part_p_, part_d_, d_sums_;
  // scratch for current_solution in fused mode
  DeviceBuffer<float> sol_a_, sol_b_, sol_c_;
};

bool BackendPDHG::plan_fused() {
  if (!opts_.fuse) return false;
  if (problem_->dualized()) return false;
  LinearOperator* K = problem_->linop();
  if (!K->all_stencil()) return false;
  if (K->blocks().size() > (size_t)kMaxFusedBlocks) return false;
  blocks_.n = 0;
  for (auto& b : K->blocks()) {
    if (b->kind() == kBlockZero) continue;       // contributes nothing
    blocks_.b[blocks_.n++] = b->desc();
  }
  auto collect = [&](const ProxList& list, std::vector<ProxDesc>& out, std::vector<ScaleRef>& scale, bool right) {
    out.clear();
    scale.clear();
    for (auto& p : list) {
      ProxDesc d;
      if (!p->leaf_desc(d, 0)) return false;
      if (dim_cap(d.dim, d.kind) == 0) return false;
      out.push_back(d);
      const size_t lo = p->index(), hi = p->index() + p->size();
      scale.push_back(right ? problem_->right_ref(lo, hi) : problem_->left_ref(lo, hi));
    }
    return true;
  };
  if (!(collect(prox_g_, g_descs_, g_scale_, true) && collect(prox_fstar_, f_descs_, f_scale_, false))) return false;
  stencil_ = opts_.fuse == 2 ? StencilPlan() : plan_stencil(K->blocks(), problem_->nrows(), problem_->ncols());
  return true;
}

void BackendPDHG::initialize(const float* h_x0, size_t nx0, const float* h_y0, size_t ny0) {
  ctx_->bind();
  if (!problem_->initialized()) fail(PB_ERR_INVALID, "Problem has not been initialized.");
  PB_TRACE_SCOPE("BackendPDHG::initialize");
  const size_t m = problem_->nrows(), n = problem_->ncols();
  cudaStream_t s = ctx_->stream;

  iteration_ = 0;
  PdhgState st{};
  st.tau = static_cast<float>(opts_.tau0);
  st.sigma = static_cast<float>(opts_.sigma0);
  st.theta = 1;
  st.arb_l = st.arb_u = 0;
  st.arg_alpha = opts_.arg_alpha0;
  st.iteration = 0;
  params_.stepsize_variant = opts_.stepsize_variant;
  params_.alg2_gamma = opts_.alg2_gamma;
  params_.arg_nu = opts_.arg_nu;
  params_.arg_delta = opts_.arg_delta;
  params_.arb_delta = opts_.arb_delta;
  params_.arb_tau = opts_.arb_tau;
  params_.tol_rel_primal = sopts_.tol_rel_primal;
  params_.tol_rel_dual = sopts_.tol_rel_dual;
  params_.tol_abs_primal = sopts_.tol_abs_primal;
  params_.tol_abs_dual = sopts_.tol_abs_dual;
  params_.nrows = m;
  params_.ncols = n;
  if (comm_) {
    // eps_primal / eps_dual (backend.hpp:71-74) are functions of the GLOBAL problem size
    double dims[2] = {static_cast<double>(m), static_cast<double>(n)};
    comm_->allreduce_sum_host(dims, 2);
    params_.nrows = static_cast<unsigned long long>(dims[0]);
    params_.ncols = static_cast<unsigned long long>(dims[1]);
  }
  st.eps_primal = pdhg_eps(params_.nrows, sopts_.tol_abs_primal, sopts_.tol_rel_primal, 0.f);
  st.eps_dual = pdhg_eps(params_.ncols, sopts_.tol_abs_dual, sopts_.tol_rel_dual, 0.f);

  // proxes, conjugated through Moreau where only the other form was given (:236-266)
  prox_g_.clear();
  prox_fstar_.clear();
  if (problem_->prox_g().empty()) {
    if (problem_->prox_gstar().empty()) fail(PB_ERR_INVALID, "Neither prox_g nor prox_gstar specified.");
    for (auto& p : problem_->prox_gstar()) prox_g_.push_back(make_prox_moreau(ctx_, p));
  } else {
    prox_g_ = problem_->prox_g();
  }
  if (problem_->prox_fstar().empty()) {
    if (problem_->prox_f().empty()) fail(PB_ERR_INVALID, "Neither prox_f nor prox_fstar specified.");
    for (auto& p : problem_->prox_f()) prox_fstar_.push_back(make_prox_moreau(ctx_, p));
  } else {
    prox_fstar_ = problem_->prox_fstar();
  }

  if (opts_.scale_steps_operator && comm_)
    fail(PB_ERR_UNSUPPORTED, "slab decomposition: scale_steps_operator (normest) is not distributed; "
                             "set scale_steps_operator = false");
  if (opts_.scale_steps_operator) {                      // :274-286
    const float norm = problem_->normest(1e-6f, 100, opts_.normest_x0);
    if (std::abs(norm - 1) > 0.1) {
      st.tau /= norm;
      st.sigma /= norm;
      if (sopts_.verbose)
        std::cout << "|K|=" << norm << " => Rescaled tau=" << st.tau << ", sigma=" << st.sigma << "."
                  << std::endl;
    }
  }

  // Slabs: a rank-local failure must not leave the peers blocked in the next collective, so every rank-local
  // verdict between two collectives is voted on (sum of failure flags) before any rank throws.
  auto vote = [&](bool ok_local, int status, const std::string& msg) {
    if (comm_) {
      double bad[1] = {ok_local ? 0.0 : 1.0};
      comm_->allreduce_sum_host(bad, 1);
      if (bad[0] != 0.0)
        fail(status, ok_local ? "slab decomposition: another rank failed to initialize (" + msg + ")" : msg);
    } else if (!ok_local) {
      fail(status, msg);
    }
  };
  vote(!(nx0 > 0 && nx0 != n), PB_ERR_INVALID, "Initial primal solution has wrong size.");
  vote(!(ny0 > 0 && ny0 != m), PB_ERR_INVALID, "Initial dual solution has wrong size.");

  { PB_TRACE_SCOPE("  plan_fused"); fused_ = plan_fused(); }
  // one-pass iterations run the ring kernel only: its dry run decides here, a launch that fails later is an error
  tile_ok_ = fused_ && opts_.fuse == 1 &&
             tile_iteration_supported(stencil_, g_descs_, f_descs_, problem_->right_ref(), problem_->left_ref()) &&
             tile_ring_available(ctx_, stencil_, g_descs_[0], f_descs_[0], comm_ != nullptr);
  // slabs: the one-pass kernel stores its edge columns straight into the neighbours' memory, so it
  // needs the peer-to-peer halo blocks
  if (comm_) tile_ok_ = tile_ok_ && stencil_.geom.nx >= 2;
  tile_iterations_ = 0;
  if (comm_) {
    // the halo protocol lives in the specialised stencil passes: one planar gradient operator
    // (+ identity rows), one prox_g over all columns, Norm2 on the gradient rows
    PrimalPass pp;                     // dry runs: is there a specialised pass for each prox?
    pp.T = problem_->right_ref();
    DualPass dp;
    dp.S = problem_->left_ref();
    bool ok = fused_ && stencil_.ok && g_descs_.size() == 1;
    if (ok) ok = stencil_primal_launch(ctx_, stencil_, g_descs_[0], pp, true) > 0;
    int halo_passes = 0;
    for (auto& d : f_descs_) {
      if (!ok) break;
      ok = stencil_dual_launch(ctx_, stencil_, d, dp, true) > 0;
      if (d.index == 0) ++halo_passes;
    }
    ok = ok && halo_passes == 1;
    // every rank must come to the same verdict, otherwise the collective below would hang
    double bad[1] = {ok ? 0.0 : 1.0};
    comm_->allreduce_sum_host(bad, 1);
    if (bad[0] != 0.0)
      fail(PB_ERR_UNSUPPORTED, "slab decomposition needs the fused stencil passes: K = planar "
                               "BlockGradient2D/3D (+ identity rows), one prox_g, Norm2 prox on the gradient rows");
    comm_->ensure_halo((size_t)stencil_.geom.ny * stencil_.geom.L);
    // all ranks run the same kind of iteration: one pass only if every slab qualifies (p2p() is only
    // known once the halo blocks are mapped)
    double no_tile[1] = {(tile_ok_ && (comm_->p2p() || comm_->world() == 1)) ? 0.0 : 1.0};
    comm_->allreduce_sum_host(no_tile, 1);
    tile_ok_ = no_tile[0] == 0.0;
  }
  {
    PB_TRACE_SCOPE("  allocate iterates");
    std::string alloc_error;
    int alloc_status = PB_OK;
    try {
      x_.resize(n); x_prev_.resize(n); y_.resize(m); y_prev_.resize(m);
      if (tile_ok_) y_stage_.resize(m);
      if (!fused_) {
        temp_.resize(std::max(m, n));
        kx_.resize(m); kx_prev_.resize(m); kty_.resize(n); kty_prev_.resize(n);
      }
      d_state_.resize(1);
      d_sums_.resize(4);
      if (tile_ok_) { fin_ticket_.resize(1); fin_ticket_.zero(s); }
    } catch (Error& e) {
      alloc_status = e.status;
      alloc_error = e.status == PB_ERR_OOM ? std::string("Out of memory: ") + e.what() : std::string(e.what());
    }
    vote(alloc_status == PB_OK, alloc_status == PB_OK ? PB_ERR_OOM : alloc_status, alloc_error.empty() ? "allocation" : alloc_error);
  }
  if (!fused_) { temp_.zero(s); kx_.zero(s); kx_prev_.zero(s); kty_.zero(s); kty_prev_.zero(s); }
  // x0 / y0 (:288-308): one host -> device copy each, the previous iterate is a device copy
  PB_TRACE_SCOPE("  x0 / y0 upload, partial buffers, state");
  if (nx0 > 0) {
    upload_from_host(ctx_, x_.data(), h_x0, n);
    PB_CUDA(cudaMemcpyAsync(x_prev_.data(), x_.data(), n * sizeof(float), cudaMemcpyDeviceToDevice, s));
  } else {
    x_.zero(s); x_prev_.zero(s);
  }
  if (ny0 > 0) {
    upload_from_host(ctx_, y_.data(), h_y0, m);
    PB_CUDA(cudaMemcpyAsync(y_prev_.data(), y_.data(), m * sizeof(float), cudaMemcpyDeviceToDevice, s));
  } else {
    y_.zero(s); y_prev_.zero(s);
  }

  // partial-sum buffers: one (a, b) pair per CTA of every launch of a pass
  if (fused_) {
    part_d_cap_ = part_p_cap_ = 0;
    // dry runs of residual-refresh passes over the iterates' buffers (the grid depends on their alignment)
    PrimalPass pp;
    pp.x = x_.data(); pp.y = y_.data(); pp.y_prev = y_prev_.data(); pp.check = true; pp.x_out = x_prev_.data();
    for (size_t i = 0; i < g_descs_.size(); ++i) {
      const ProxDesc& d = g_descs_[i];
      pp.T = g_scale_[i];
      part_d_cap_ += std::max(stencil_primal_launch(ctx_, stencil_, d, pp, true), fused_grid(ctx_, d));
    }
    DualPass dp;
    dp.y = y_.data(); dp.x_new = x_.data(); dp.x_old = x_prev_.data(); dp.check = true; dp.y_out = y_prev_.data();
    for (size_t i = 0; i < f_descs_.size(); ++i) {
      const ProxDesc& d = f_descs_[i];
      dp.S = f_scale_[i];
      part_p_cap_ += std::max(stencil_dual_launch(ctx_, stencil_, d, dp, true), fused_grid(ctx_, d));
    }
  } else {
    part_p_cap_ = std::min<size_t>(grid_for(m), (size_t)ctx_->num_sms * 8);
    part_d_cap_ = std::min<size_t>(grid_for(n), (size_t)ctx_->num_sms * 8);
  }
  part_p_.resize(2 * (size_t)std::max(part_p_cap_, 1u));
  part_d_.resize(2 * (size_t)std::max(part_d_cap_, 1u));

  h_state_ = st;
  d_state_.upload(&h_state_, 1, s);
  PB_CUDA(cudaStreamSynchronize(s));
}

void BackendPDHG::iteration_fused() {
  const bool check = is_check_iteration();
  const ScaleRef T = problem_->right_ref(), S = problem_->left_ref();
  const PdhgState* st = d_state_.data();

  unsigned nd = 0, np = 0;
  const bool tiled = tile_ok_ && iteration_ > 0;
  const RingHalo ring_halo = tiled && comm_ ? comm_->ring_halo() : RingHalo();
  bool finished_in_kernel = false;
  if (tiled) {
    // whole iteration in one pass over HBM (pb_tile.cu): x_prev_ <- x^{k+1}, y_prev_ <- y^{k+1}
    TilePass tp;
    tp.x = x_.data(); tp.y = y_.data(); tp.T = T; tp.S = S; tp.st = st; tp.x_out = x_prev_.data();
    tp.y_out = y_prev_.data();
    tp.halo = comm_ ? &ring_halo : nullptr;
    RingFinish fin;
    if (check) {
      // the residual-refresh launch folds the sums, combines them across ranks and advances the step-size state
      // itself (RingFinish) unless the halos travel through NCCL staging buffers (no peer-mapped slots then)
      finished_in_kernel = !comm_ || comm_->world() == 1 || comm_->reduce_p2p();
      if (finished_in_kernel) { fin = ring_finish(); tp.finish = &fin; }
      tp.check = true;
      tp.y_prev = y_prev_.data();
      tp.ktyprev_zero = iteration_ <= 1;
      tp.part_d = part_d_.data(); tp.part_p = part_p_.data();
      // y^{k+1} cannot overwrite y_prev_ (the pass reads y^{k-1} from it), so it goes to a third buffer that
      // then takes y_prev_'s place
      tp.y_out = y_prev_staging();
    }
    nd = np = tile_iteration_launch(ctx_, stencil_, g_descs_[0], f_descs_[0], tp);
    x_.swap(x_prev_);
    if (check) {
      y_prev_.swap(y_stage_);    // y_prev_ now holds y^{k+1}, y_stage_ the dead y^{k-1}
      tile_check_iterations_++;
    }
    y_.swap(y_prev_);            // y_ = y^{k+1}, y_prev_ = y^k
    tile_iterations_++;
    if (prof_ev_) {
      PB_CUDA(cudaEventRecord(prof_ev_[1], ctx_->stream));
      PB_CUDA(cudaEventRecord(prof_ev_[2], ctx_->stream));
    }
  } else {
    // primal pass: x_prev_ <- prox_g(x_ - tau T K^T y_), then swap so that x_ is x^{k+1}.  Each prox range runs
    // the specialised stencil pass where one covers it, the generic fused pass otherwise.
    unsigned off = 0;
    const SlabHalo primal_halo = comm_ ? comm_->primal_halo() : SlabHalo();
    PrimalPass pp;
    pp.x = x_.data(); pp.y = y_.data(); pp.y_prev = y_prev_.data(); pp.st = st;
    pp.kty_zero = iteration_ == 0; pp.ktyprev_zero = iteration_ <= 1; pp.check = check;
    pp.x_out = x_prev_.data();
    pp.halo = comm_ ? &primal_halo : nullptr;
    for (size_t i = 0; i < g_descs_.size(); ++i) {
      const ProxDesc& d = g_descs_[i];
      pp.T = g_scale_[i];
      pp.partials = part_d_.data() + 2 * (size_t)off;
      unsigned g = stencil_primal_launch(ctx_, stencil_, d, pp);
      if (g == 0) g = fused_primal_launch(ctx_, d, blocks_, pp);
      off += g;
    }
    nd = off;
    x_.swap(x_prev_);
    const SlabHalo dual_halo = comm_ ? comm_->dual_halo() : SlabHalo();
    if (prof_ev_) PB_CUDA(cudaEventRecord(prof_ev_[1], ctx_->stream));

    // dual pass: y_prev_ <- prox_f*(y_ + sigma S K(2x^{k+1} - x^k)) (theta-extrapolated), then swap
    off = 0;
    DualPass dp;
    dp.y = y_.data(); dp.x_new = x_.data(); dp.x_old = x_prev_.data(); dp.st = st;
    dp.kxprev_zero = iteration_ == 0; dp.check = check;
    dp.y_out = y_prev_.data();
    dp.halo = comm_ ? &dual_halo : nullptr;
    for (size_t i = 0; i < f_descs_.size(); ++i) {
      const ProxDesc& d = f_descs_[i];
      dp.S = f_scale_[i];
      dp.partials = part_p_.data() + 2 * (size_t)off;
      unsigned g = stencil_dual_launch(ctx_, stencil_, d, dp);
      if (g == 0) g = fused_dual_launch(ctx_, d, blocks_, dp);
      off += g;
    }
    np = off;
    y_.swap(y_prev_);
    // with tile_ok_ this is iteration 0 of a ROF-shaped slab problem: the one-pass iterations that follow read the
    // halo columns it received from the flag-in-data slots
    if (comm_) comm_->end_two_pass_iteration(tile_ok_);
    if (prof_ev_) PB_CUDA(cudaEventRecord(prof_ev_[2], ctx_->stream));

  }
  if (finished_in_kernel) {
    // nothing to launch: residual sums, cross-rank combination and pdhg_update happened in the ring kernel
  } else if (comm_ && comm_->world() > 1 && check) {
    // per-rank fold -> one 4-double all-reduce -> identical state machine on every rank
    fold_residuals_kernel<<<1, kBlock, 0, ctx_->stream>>>(part_p_.data(), np, part_d_.data(), nd,
                                                          d_sums_.data());
    PB_CHECK_LAUNCH();
    comm_->allreduce_sum(d_sums_.data(), 4);
    pdhg_finalize_sums_kernel<<<1, 32, 0, ctx_->stream>>>(d_state_.data(), params_, d_sums_.data(),
                                                          iteration_, 1);
    PB_CHECK_LAUNCH();
    ctx_->launches += 2;
  } else if (check || opts_.stepsize_variant == PB_PDHG_ALG2) {
    pdhg_finalize_kernel<<<1, kBlock, 0, ctx_->stream>>>(d_state_.data(), params_, part_p_.data(), np,
                                                         part_d_.data(), nd, iteration_, check ? 1 : 0);
    PB_CHECK_LAUNCH();
    ctx_->launches++;
  }
  iteration_++;
}

RingFinish BackendPDHG::ring_finish() {
  RingFinish f;
  f.ticket = fin_ticket_.data();
  f.state = d_state_.data();
  f.prm = params_;
  f.iteration = iteration_;
  if (comm_ && comm_->world() > 1) f.cross = comm_->cross_sum();
  return f;
}

// K u / K^T p on the local slab including the neighbours' columns (current_solution only)
void BackendPDHG::slab_apply(float* d_res, const float* d_rhs, const float* d_halo, bool adjoint) {
  GradGeom g = stencil_.geom;
  g.q = g.ny;
  g.div_q = FastDiv(g.ny);
  g.div_nx = FastDiv(g.nx);
  g.halo = SlabHalo();
  g.halo.has_left = comm_->has_left();
  g.halo.has_right = comm_->has_right();
  const unsigned grid = (g.plane + kStencilBlock - 1) / kStencilBlock;
  cudaStream_t s = ctx_->stream;
  if (!adjoint) {
    if (stencil_.three_d) slab_forward_kernel<true><<<grid, kStencilBlock, 0, s>>>(g, d_rhs, d_halo, d_res);
    else slab_forward_kernel<false><<<grid, kStencilBlock, 0, s>>>(g, d_rhs, d_halo, d_res);
  } else if (stencil_.three_d) {
    if (g.has_id) slab_adjoint_kernel<true, true><<<grid, kStencilBlock, 0, s>>>(g, d_rhs, d_halo, d_res);
    else slab_adjoint_kernel<true, false><<<grid, kStencilBlock, 0, s>>>(g, d_rhs, d_halo, d_res);
  } else {
    if (g.has_id) slab_adjoint_kernel<false, true><<<grid, kStencilBlock, 0, s>>>(g, d_rhs, d_halo, d_res);
    else slab_adjoint_kernel<false, false><<<grid, kStencilBlock, 0, s>>>(g, d_rhs, d_halo, d_res);
  }
  PB_CHECK_LAUNCH();
}

void BackendPDHG::iteration_unfused() {
  const size_t m = problem_->nrows(), n = problem_->ncols();
  cudaStream_t s = ctx_->stream;
  const float* T = problem_->scaling_right();
  const float* S = problem_->scaling_left();
  PdhgState& st = h_state_;

  primal_proxarg_kernel<<<sgrid(n), kBlock, 0, s>>>(temp_.data(), x_.data(), T, kty_.data(), n, st.tau);
  PB_CHECK_LAUNCH();
  x_.swap(x_prev_);
  for (auto& p : prox_g_) p->eval(x_.data(), temp_.data(), T, st.tau, false);
  kx_.swap(kx_prev_);
  problem_->apply_K(kx_.data(), x_.data(), false);
  dual_proxarg_kernel<<<sgrid(m), kBlock, 0, s>>>(temp_.data(), y_.data(), S, kx_.data(), kx_prev_.data(),
                                                  m, st.sigma, st.theta);
  PB_CHECK_LAUNCH();
  y_.swap(y_prev_);
  for (auto& p : prox_fstar_) p->eval(y_.data(), temp_.data(), S, st.sigma, false);
  ctx_->launches += 2;

  const bool check = is_check_iteration();
  double sums[4] = {0, 0, 0, 0};
  if (check) {
    primal_residual_kernel<<<part_p_cap_, kBlock, 0, s>>>(y_prev_.data(), y_.data(), S, kx_prev_.data(),
                                                          kx_.data(), m, st.sigma, st.theta, part_p_.data());
    PB_CHECK_LAUNCH();
    dual_residual_kernel<<<part_d_cap_, kBlock, 0, s>>>(x_prev_.data(), x_.data(), T, kty_prev_.data(),
                                                        kty_.data(), n, st.tau, part_d_.data());
    PB_CHECK_LAUNCH();
    fold_residuals_kernel<<<1, kBlock, 0, s>>>(part_p_.data(), part_p_cap_, part_d_.data(), part_d_cap_,
                                               d_sums_.data());
    PB_CHECK_LAUNCH();
    ctx_->launches += 3;
    d_sums_.download(sums, 4, s);
    PB_CUDA(cudaStreamSynchronize(s));
  }
  st.iteration = iteration_;
  pdhg_update(st, params_, sums, check);
  iteration_++;

  kty_.swap(kty_prev_);
  problem_->apply_K(kty_.data(), y_.data(), true);
}

void BackendPDHG::profile(int n_iters, float out_ms[3]) {
  float d[8];
  profile_detail(n_iters, d);
  // averages over ALL profiled iterations (tiled iterations count as "primal pass" time)
  const float n2 = d[4], nt = d[5], nc = d[7], n = n2 + nt + nc;
  out_ms[0] = n > 0 ? (d[0] * n2 + d[3] * nt + d[6] * nc) / n : 0.f;
  out_ms[1] = n > 0 ? d[1] * n2 / n : 0.f;
  out_ms[2] = n > 0 ? d[2] : 0.f;
}

// out = { primal pass ms, dual pass ms (both averaged over the two-pass iterations), finalize ms
// (averaged over all), tiled whole-iteration kernel ms (averaged over the tiled iterations that do not
// refresh the residuals), number of two-pass iterations, number of such tiled iterations, tiled
// residual-refresh kernel ms, number of tiled residual-refresh iterations }
void BackendPDHG::profile_detail(int n_iters, float out[8]) {
  ctx_->bind();
  for (int k = 0; k < 8; ++k) out[k] = 0.f;
  if (!fused_ || n_iters <= 0) { iterate(n_iters); return; }
  // four events per iteration, all recorded back to back and read after ONE synchronisation at the end: the
  // iterations run exactly as in iterate() (no host round trip between them, so on slabs no rank skew either)
  std::vector<cudaEvent_t> ev(4 * (size_t)n_iters);
  for (auto& e : ev) PB_CUDA(cudaEventCreate(&e));
  std::vector<unsigned char> kind(n_iters);          // 0 two-pass, 1 one-pass, 2 one-pass with residual refresh
  for (int i = 0; i < n_iters; ++i) {
    const unsigned long long tiles_before = tile_iterations_, chk_before = tile_check_iterations_;
    prof_ev_ = &ev[4 * (size_t)i];
    PB_CUDA(cudaEventRecord(prof_ev_[0], ctx_->stream));
    iteration_fused();
    PB_CUDA(cudaEventRecord(prof_ev_[3], ctx_->stream));
    kind[i] = tile_check_iterations_ != chk_before ? 2 : (tile_iterations_ != tiles_before ? 1 : 0);
  }
  prof_ev_ = nullptr;
  PB_CUDA(cudaStreamSynchronize(ctx_->stream));
  double acc[5] = {0, 0, 0, 0, 0};
  int n_two = 0, n_tile = 0, n_chk = 0;
  for (int i = 0; i < n_iters; ++i) {
    float ms[3];
    for (int k = 0; k < 3; ++k) PB_CUDA(cudaEventElapsedTime(&ms[k], ev[4 * (size_t)i + k], ev[4 * (size_t)i + k + 1]));
    if (kind[i] == 2) { acc[4] += ms[0]; ++n_chk; }
    else if (kind[i] == 1) { acc[3] += ms[0]; ++n_tile; }
    else { acc[0] += ms[0]; acc[1] += ms[1]; ++n_two; }
    acc[2] += ms[2];
  }
  for (auto& e : ev) cudaEventDestroy(e);
  out[0] = n_two ? static_cast<float>(acc[0] / n_two) : 0.f;
  out[1] = n_two ? static_cast<float>(acc[1] / n_two) : 0.f;
  out[2] = static_cast<float>(acc[2] / n_iters);
  out[3] = n_tile ? static_cast<float>(acc[3] / n_tile) : 0.f;
  out[4] = static_cast<float>(n_two);
  out[5] = static_cast<float>(n_tile);
  out[6] = n_chk ? static_cast<float>(acc[4] / n_chk) : 0.f;
  out[7] = static_cast<float>(n_chk);
}

void BackendPDHG::iterate(int n_iters) {
  ctx_->bind();
  for (int i = 0; i < n_iters; ++i) {
    if (fused_) iteration_fused();
    else iteration_unfused();
  }
}

PdhgState BackendPDHG::fetch_state() {
  if (fused_) {
    d_state_.download(&h_state_, 1, ctx_->stream);
    PB_CUDA(cudaStreamSynchronize(ctx_->stream));
  }
  return h_state_;
}

void BackendPDHG::residuals(float out[6]) {
  ctx_->bind();
  const PdhgState st = fetch_state();
  if (comm_) comm_->check_error();
  out[0] = st.primal_residual;
  out[1] = st.dual_residual;
  out[2] = st.primal_var_norm;
  out[3] = st.dual_var_norm;
  out[4] = st.eps_primal;
  out[5] = st.eps_dual;
  if (!comm_) {
    // Backend::eps_primal() / eps_dual() are evaluated at call time with the problem's CURRENT dimensions
    // (backend.hpp:71-74): once a dualised solve has been restored (solver.cu:199-203) those are the original
    // ones again, which is what a caller reading them after Solver::Solve() gets from the reference
    out[4] = pdhg_eps(problem_->nrows(), sopts_.tol_abs_primal, sopts_.tol_rel_primal, st.primal_var_norm);
    out[5] = pdhg_eps(problem_->ncols(), sopts_.tol_abs_dual, sopts_.tol_rel_dual, st.dual_var_norm);
  }
}

void BackendPDHG::stepsizes(double out[3]) {
  ctx_->bind();
  const PdhgState st = fetch_state();
  out[0] = st.tau;
  out[1] = st.sigma;
  out[2] = st.theta;
}

void BackendPDHG::current_solution(float* h_x, float* h_z, float* h_y, float* h_w) {
  ctx_->bind();
  const size_t m = problem_->nrows(), n = problem_->ncols();
  cudaStream_t s = ctx_->stream;
  const PdhgState st = fetch_state();
  PB_TRACE_SCOPE("BackendPDHG::current_solution");
  if (h_x) download_to_host(ctx_, h_x, x_.data(), n);
  if (h_y) download_to_host(ctx_, h_y, y_.data(), m);
  if (h_w || h_z) {
    const ScaleRef T = problem_->right_ref(), S = problem_->left_ref();
    if (fused_) {
      // K x, K x_prev and K^T y_prev are not stored in fused mode: rebuild them with the
      // unfused operator, honouring the zero-initialised history of the reference
      const Comm::PlainHalo halo = comm_ ? comm_->plain_halo() : Comm::PlainHalo();
      if (h_w) {
        const size_t cap = std::max(n, m);       // one allocation serves w (n) and z (m)
        if (sol_a_.size() != cap) { sol_a_.resize(cap); sol_b_.resize(cap); }
        if (iteration_ <= 1) PB_CUDA(cudaMemsetAsync(sol_a_.data(), 0, n * sizeof(float), s));
        else if (comm_) slab_apply(sol_a_.data(), y_prev_.data(), halo.y_prev, true);
        else problem_->apply_K(sol_a_.data(), y_prev_.data(), true);
        w_variable_kernel<<<sgrid(n), kBlock, 0, s>>>(sol_b_.data(), x_prev_.data(), x_.data(), T,
                                                      sol_a_.data(), n, st.tau);
        PB_CHECK_LAUNCH();
        download_to_host(ctx_, h_w, sol_b_.data(), n);
      }
      if (h_z) {
        const size_t cap = std::max(n, m);
        if (sol_a_.size() != cap) { sol_a_.resize(cap); sol_b_.resize(cap); }
        if (sol_c_.size() != m) sol_c_.resize(m);
        if (iteration_ == 0) PB_CUDA(cudaMemsetAsync(sol_a_.data(), 0, m * sizeof(float), s));
        else if (comm_) slab_apply(sol_a_.data(), x_.data(), halo.x, false);
        else problem_->apply_K(sol_a_.data(), x_.data(), false);
        if (iteration_ <= 1) PB_CUDA(cudaMemsetAsync(sol_b_.data(), 0, m * sizeof(float), s));
        else if (comm_) slab_apply(sol_b_.data(), x_prev_.data(), halo.x_prev, false);
        else problem_->apply_K(sol_b_.data(), x_prev_.data(), false);
        z_variable_kernel<<<sgrid(m), kBlock, 0, s>>>(sol_c_.data(), y_prev_.data(), y_.data(), S,
                                                      sol_a_.data(), sol_b_.data(), m, st.sigma, st.theta);
        PB_CHECK_LAUNCH();
        download_to_host(ctx_, h_z, sol_c_.data(), m);
      }
    } else {
      if (h_w) {
        w_variable_kernel<<<sgrid(n), kBlock, 0, s>>>(temp_.data(), x_prev_.data(), x_.data(), T,
                                                      kty_prev_.data(), n, st.tau);
        PB_CHECK_LAUNCH();
        download_to_host(ctx_, h_w, temp_.data(), n);
      }
      if (h_z) {
        z_variable_kernel<<<sgrid(m), kBlock, 0, s>>>(temp_.data(), y_prev_.data(), y_.data(), S,
                                                      kx_.data(), kx_prev_.data(), m, st.sigma, st.theta);
        PB_CHECK_LAUNCH();
        download_to_host(ctx_, h_z, temp_.data(), m);
      }
    }
  }
  PB_CUDA(cudaStreamSynchronize(s));
  // slab mode: the halo slots read above are overwritten by the neighbours' next passes, so no rank
  // may run ahead before every rank is done reading (current_solution is collective)
  if (comm_) { comm_->check_error(); comm_->barrier(); }
}

std::shared_ptr<Backend> make_backend_pdhg(Context* ctx, std::shared_ptr<Problem> prob,
                                           const pb_pdhg_options& opts, const pb_solver_options& sopts) {
  return std::make_shared<BackendPDHG>(ctx, std::move(prob), opts, sopts);
}

}  // namespace pb
