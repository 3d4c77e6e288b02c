// pb_problem.cuh -- Problem (graph-form problem container): include/prost/problem.hpp:64-114,
// src/problem.cu.
#pragma once

#include <functional>
#include <memory>
#include <string>
#include <vector>

#include "pb_linop.cuh"
#include "pb_prox.cuh"

namespace pb {

typedef std::vector<std::shared_ptr<Prox>> ProxList;

// One diagonal preconditioner (Sigma or T).  Gradient-type operators give piecewise-constant -- for a
// single block constant -- preconditioners, so the vector is kept as a few (begin, end, value) segments
// and only materialised (host vector / device vector) for the consumers that index it per element.
// The reference builds both vectors element by element through two virtual calls per row and column
// (problem.cu:262-287) and uploads them; at 4096^2 that was 0.3 s of a 0.9 s solve here.
struct ScaleSeg { size_t begin, end; float value; };
class ScaleVec {
 public:
  void set_segments(size_t n, std::vector<ScaleSeg> segs);
  void set_host(std::vector<float> v);
  size_t size() const { return n_; }
  bool uniform() const { return uniform_; }
  float value() const { return value_; }                 // meaningful when uniform()
  bool has_segments() const { return !segs_.empty() || n_ == 0; }
  const std::vector<ScaleSeg>& segments() const { return segs_; }
  const std::vector<float>& host() const;                // materialises on first use
  const float* device(Context* ctx) const;               // materialises on first use
  // scalar when every entry of [begin, end) has the same value (one segment), else the device vector
  ScaleRef ref(Context* ctx, size_t begin, size_t end) const;
  void swap(ScaleVec& o);

 private:
  size_t n_ = 0;
  bool uniform_ = false;
  float value_ = 1.f;
  std::vector<ScaleSeg> segs_;                           // empty: only the host vector is authoritative
  mutable std::vector<float> host_;
  mutable bool host_valid_ = false;
  mutable DeviceBuffer<float> dev_;
  mutable bool dev_valid_ = false;
};

class Comm;

// K / K^T and the sum over ranks of the power iteration (Problem::normest); empty members: the problem's own
// operator (apply_K) on one GPU
struct NormestOps {
  std::function<void(float* d_res, const float* d_rhs, bool adjoint)> apply;
  std::function<void(double* h_buf, size_t n)> sum;
};

class Problem {
 public:
  enum Scaling { kScalingIdentity, kScalingAlpha, kScalingCustom };

  explicit Problem(Context* ctx) : ctx_(ctx), linop_(new LinearOperator(ctx)) {}

  void add_block(std::shared_ptr<Block> b) { linop_->add_block(std::move(b)); }
  void add_prox_g(std::shared_ptr<Prox> p) { prox_g_.push_back(std::move(p)); }
  void add_prox_f(std::shared_ptr<Prox> p) { prox_f_.push_back(std::move(p)); }
  void add_prox_gstar(std::shared_ptr<Prox> p) { prox_gstar_.push_back(std::move(p)); }
  void add_prox_fstar(std::shared_ptr<Prox> p) { prox_fstar_.push_back(std::move(p)); }
  void set_dimensions(size_t nrows, size_t ncols) { nrows_ = nrows; ncols_ = ncols; dims_set_ = true; }
  void set_scaling_alpha(float alpha) { scaling_type_ = kScalingAlpha; scaling_alpha_ = alpha; }
  void set_scaling_identity() { scaling_type_ = kScalingIdentity; }
  Scaling scaling_type() const { return scaling_type_; }
  void set_scaling_custom(const float* left, size_t nl, const float* right, size_t nr);

  void initialize();
  // Row shards (BackendADMM): after initialize() on this rank's rows, replace the alpha preconditioners by those
  // of the whole operator -- T from the column sums over all ranks' rows, and Sigma and T with the empty-row /
  // empty-column carry running across the ranks in rank order.  Collective.
  void shard_alpha_scaling(Comm& comm);
  void dualize();
  // on a slab (rank-local problem) only with `ops` that apply the global operator; h_x0: ncols floats or NULL
  float normest(float tol, int max_iters, const float* h_x0, const NormestOps& ops = NormestOps());

  size_t nrows() const { return nrows_; }
  size_t ncols() const { return ncols_; }
  size_t gpu_mem_amount() const;
  bool dualized() const { return dualized_; }
  bool initialized() const { return initialized_; }

  LinearOperator* linop() const { return linop_.get(); }
  // K apply honouring Dualize(): primal problem K / K^T, dual problem -K^T / -K
  void apply_K(float* d_res, const float* d_rhs, bool adjoint);

  const ProxList& prox_g() const { return prox_g_; }
  const ProxList& prox_f() const { return prox_f_; }
  const ProxList& prox_gstar() const { return prox_gstar_; }
  const ProxList& prox_fstar() const { return prox_fstar_; }

  // Sigma (left, nrows) and T (right, ncols)
  const float* scaling_left() const { return left_.device(ctx_); }
  const float* scaling_right() const { return right_.device(ctx_); }
  const std::vector<float>& scaling_left_host() const { return left_.host(); }
  const std::vector<float>& scaling_right_host() const { return right_.host(); }
  ScaleRef left_ref() const { return left_.uniform() ? ScaleRef{nullptr, left_.value()} : ScaleRef{left_.device(ctx_), 1.f}; }
  ScaleRef right_ref() const { return right_.uniform() ? ScaleRef{nullptr, right_.value()} : ScaleRef{right_.device(ctx_), 1.f}; }
  // the same for the index range of one prox: gradient rows and identity rows of a stacked operator have
  // different, but per range constant, preconditioners -- the fused passes then read no Sigma / T at all
  ScaleRef left_ref(size_t begin, size_t end) const { return left_.ref(ctx_, begin, end); }
  ScaleRef right_ref(size_t begin, size_t end) const { return right_.ref(ctx_, begin, end); }
  Context* ctx() const { return ctx_; }

 private:
  void average_preconditioners(std::vector<float>& precond, const ProxList& prox);
  bool scaling_segments(std::vector<ScaleSeg>& left, std::vector<ScaleSeg>& right) const;
  static bool average_segments(std::vector<ScaleSeg>& segs, const ProxList& prox);

  Context* ctx_;
  std::shared_ptr<LinearOperator> linop_;
  ProxList prox_g_, prox_f_, prox_gstar_, prox_fstar_;
  size_t nrows_ = 0, ncols_ = 0;
  bool dims_set_ = false;
  // the reference leaves scaling_type_ uninitialised in C++ (problem.hpp:125); MATLAB always
  // sets alpha = 1 (matlab/+prost/problem.m:10), which is the default here (Appendix B #19)
  Scaling scaling_type_ = kScalingAlpha;
  float scaling_alpha_ = 1.f;
  std::vector<float> custom_left_, custom_right_;       // SetScalingCustom (squares of the user vectors)
  ScaleVec left_, right_;
  bool dualized_ = false;
  bool initialized_ = false;
};

}  // namespace pb
