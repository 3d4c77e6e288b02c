// pb_problem.cu -- Problem::Initialize (prox domain checks, zero-prox fill, Pock-Chambolle
// diagonal preconditioning, preconditioner averaging), normest and Dualize.
// Reference: src/problem.cu:47-158 (domain), :195-323 (Initialize), :428-500 (normest),
// :502-536 (AveragePreconditioners), :538-547 (Dualize).
#include "pb_problem.cuh"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <iostream>

#include "pb_comm.cuh"
#include "pb_reduce.cuh"

namespace pb {

// ---- small kernels for normest -------------------------------------------------------------------

// out = sqrt(scale) * in   (normest_multiplies_sqrt, problem.cu:417-426)
__global__ void __launch_bounds__(kBlock) mul_sqrt_kernel(float* __restrict__ out,
                                                          const float* __restrict__ scale,
                                                          const float* __restrict__ in, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x)
    out[i] = sqrtf(scale[i]) * in[i];
}

__global__ void __launch_bounds__(kBlock) divide_kernel(float* __restrict__ v, size_t n, float fac) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x)
    v[i] = v[i] / fac;
}

__global__ void __launch_bounds__(kBlock) sumsq_partial_kernel(const float* __restrict__ v, size_t n,
                                                               double* __restrict__ part) {
  double a = 0.0, b = 0.0;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x) {
    const float x = v[i];
    a += static_cast<double>(x * x);
  }
  block_sum2(a, b);
  if (threadIdx.x == 0) { part[2 * blockIdx.x] = a; part[2 * blockIdx.x + 1] = 0.0; }
}

__global__ void __launch_bounds__(kBlock) fold_kernel(const double* __restrict__ part, unsigned n,
                                                      double* __restrict__ out) {
  double a, b;
  fold_partials2(part, n, a, b);
  if (threadIdx.x == 0) { out[0] = a; out[1] = b; }
}

static double device_sumsq(Context* ctx, const float* v, size_t n, DeviceBuffer<double>& scratch) {
  const unsigned grid = std::min<size_t>(grid_for(n), (size_t)ctx->num_sms * 8);
  if (scratch.size() < 2 * (size_t)grid + 2) scratch.resize(2 * (size_t)grid + 2);
  sumsq_partial_kernel<<<grid, kBlock, 0, ctx->stream>>>(v, n, scratch.data() + 2);
  PB_CHECK_LAUNCH();
  fold_kernel<<<1, kBlock, 0, ctx->stream>>>(scratch.data() + 2, grid, scratch.data());
  PB_CHECK_LAUNCH();
  ctx->launches += 2;
  double h[2];
  PB_CUDA(cudaMemcpyAsync(h, scratch.data(), sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  PB_CUDA(cudaStreamSynchronize(ctx->stream));
  return h[0];
}

// ---- domain checks ---------------------------------------------------------------------------------

static ProxList sorted_by_index(const ProxList& proxs) {
  ProxList s = proxs;
  std::sort(s.begin(), s.end(), [](const std::shared_ptr<Prox>& a, const std::shared_ptr<Prox>& b) {
    return a->index() < b->index();
  });
  return s;
}

// AddZeroProx (problem.cu:92-158): fill uncovered index ranges with identity proxes
static void add_zero_prox(Context* ctx, ProxList& proxs, size_t n, const std::string& name) {
  if (proxs.empty()) return;
  ProxList s = sorted_by_index(proxs);
  if (s[0]->index() > 0) proxs.push_back(make_prox_zero(ctx, 0, s[0]->index()));
  for (size_t i = 0; i + 1 < s.size(); ++i) {
    if (s[i]->end() + 1 < s[i + 1]->index()) {
      const size_t start = s[i]->end() + 1;
      proxs.push_back(make_prox_zero(ctx, start, s[i + 1]->index() - start));
    }
  }
  const auto& last = s.back();
  if (last->end() != n - 1) {
    if (last->end() < n - 1) {
      const size_t start = last->end() + 1;
      proxs.push_back(make_prox_zero(ctx, start, (n - 1) - last->end()));
    } else {
      std::ostringstream ss;
      ss << name << " (AddZeroProx): Last prox operator ends after the domain: [" << last->index()
         << ", " << last->end() << "], end = " << n - 1 << "." << std::endl;
      fail(PB_ERR_INVALID, ss.str());
    }
  }
}

// CheckDomainProx (problem.cu:47-89)
static void check_domain_prox(const ProxList& proxs, size_t n, const std::string& name) {
  if (proxs.empty()) return;
  ProxList s = sorted_by_index(proxs);
  for (size_t i = 0; i + 1 < s.size(); ++i) {
    if (s[i]->end() != s[i + 1]->index() - 1) {
      std::ostringstream ss;
      ss << name << " (CheckDomainProx): Prox operators are overlapping: [" << s[i]->index() << ", "
         << s[i]->end() << "] and [" << s[i + 1]->index() << ", " << s[i + 1]->end() << "]." << std::endl;
      fail(PB_ERR_INVALID, ss.str());
    }
  }
  const auto& last = s.back();
  if (last->end() != n - 1) {
    std::ostringstream ss;
    ss << name << " (CheckDomainProx): Last prox operator "
       << (last->end() < n - 1 ? "ends too early: [" : "ends after the domain: [") << last->index()
       << ", " << last->end() << "], end = " << n - 1 << "." << std::endl;
    fail(PB_ERR_INVALID, ss.str());
  }
}

// ---- Problem ---------------------------------------------------------------------------------------

void Problem::set_scaling_custom(const float* left, size_t nl, const float* right, size_t nr) {
  scaling_type_ = kScalingCustom;
  // the reference stores the SQUARES of the user vectors (problem.cu:344-364)
  custom_left_.resize(nl);
  custom_right_.resize(nr);
  for (size_t i = 0; i < nl; ++i) custom_left_[i] = left[i] * left[i];
  for (size_t i = 0; i < nr; ++i) custom_right_[i] = right[i] * right[i];
}

// ---- ScaleVec ---------------------------------------------------------------------------------------

__global__ void __launch_bounds__(kBlock) fill_range_kernel(float* __restrict__ v, size_t n, float value) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    v[i] = value;
}

void ScaleVec::set_segments(size_t n, std::vector<ScaleSeg> segs) {
  n_ = n;
  segs_.clear();
  for (auto& s : segs) {                       // merge neighbours with equal values
    if (s.begin >= s.end) continue;
    if (!segs_.empty() && segs_.back().end == s.begin && segs_.back().value == s.value) segs_.back().end = s.end;
    else segs_.push_back(s);
  }
  uniform_ = n == 0 || (segs_.size() == 1 && segs_[0].begin == 0 && segs_[0].end == n);
  value_ = segs_.empty() ? 1.f : segs_[0].value;
  host_.clear(); host_.shrink_to_fit();
  host_valid_ = dev_valid_ = false;
  dev_.release();
}

void ScaleVec::set_host(std::vector<float> v) {
  n_ = v.size();
  segs_.clear();
  host_ = std::move(v);
  host_valid_ = true;
  dev_valid_ = false;
  dev_.release();
  uniform_ = true;
  for (size_t i = 1; i < n_ && uniform_; ++i) uniform_ = host_[i] == host_[0];
  value_ = n_ ? host_[0] : 1.f;
}

const std::vector<float>& ScaleVec::host() const {
  if (!host_valid_) {
    host_.resize(n_);
    for (auto& s : segs_) std::fill(host_.begin() + s.begin, host_.begin() + s.end, s.value);
    host_valid_ = true;
  }
  return host_;
}

const float* ScaleVec::device(Context* ctx) const {
  if (!dev_valid_) {
    dev_.resize(n_);
    if (!segs_.empty()) {
      for (auto& s : segs_) {
        const size_t len = s.end - s.begin;
        const unsigned grid = (unsigned)std::min<size_t>(grid_for(len), (size_t)ctx->num_sms * 16);
        fill_range_kernel<<<grid, kBlock, 0, ctx->stream>>>(dev_.data() + s.begin, len, s.value);
        PB_CHECK_LAUNCH();
      }
    } else if (n_) {
      upload_from_host(ctx, dev_.data(), host_.data(), n_);
    }
    dev_valid_ = true;
  }
  return dev_.data();
}

ScaleRef ScaleVec::ref(Context* ctx, size_t begin, size_t end) const {
  if (uniform_) return ScaleRef{nullptr, value_};
  for (auto& s : segs_)
    if (s.begin <= begin && begin < s.end && end <= s.end) return ScaleRef{nullptr, s.value};
  return ScaleRef{device(ctx), 1.f};
}

void ScaleVec::swap(ScaleVec& o) {
  std::swap(n_, o.n_);
  std::swap(uniform_, o.uniform_);
  std::swap(value_, o.value_);
  segs_.swap(o.segs_);
  host_.swap(o.host_);
  std::swap(host_valid_, o.host_valid_);
  dev_.swap(o.dev_);
  std::swap(dev_valid_, o.dev_valid_);
}

// Pock-Chambolle preconditioners in segment form: possible when every block has index-independent
// row / column sums (gradient and zero blocks).  Same arithmetic as the element-wise loop in
// Problem::initialize: float sum over the blocks in list order, 1. / s in double, empty rows / columns
// carry the previous value, and the carry runs from the last row into the first column.
bool Problem::scaling_segments(std::vector<ScaleSeg>& left, std::vector<ScaleSeg>& right) const {
  const auto& blocks = linop_->blocks();
  if (blocks.size() > 64) return false;
  for (auto& b : blocks)
    if (!b->uniform_sums()) return false;
  float value = 1;
  auto build = [&](bool rows, size_t n, float alpha, std::vector<ScaleSeg>& out) {
    std::vector<size_t> cuts = {0, n};
    for (auto& b : blocks) {
      const size_t lo = rows ? b->row() : b->col(), hi = lo + (rows ? b->nrows() : b->ncols());
      cuts.push_back(std::min(lo, n));
      cuts.push_back(std::min(hi, n));
    }
    std::sort(cuts.begin(), cuts.end());
    cuts.erase(std::unique(cuts.begin(), cuts.end()), cuts.end());
    for (size_t k = 0; k + 1 < cuts.size(); ++k) {
      float sum = 0.f;
      for (auto& b : blocks) {
        const size_t lo = rows ? b->row() : b->col(), len = rows ? b->nrows() : b->ncols();
        if (len && cuts[k] >= lo && cuts[k] < lo + len) sum += rows ? b->row_sum(0, alpha) : b->col_sum(0, alpha);
      }
      if (sum > 0) value = static_cast<float>(1. / sum);
      out.push_back({cuts[k], cuts[k + 1], value});
    }
  };
  build(true, nrows_, scaling_alpha_, left);
  build(false, ncols_, static_cast<float>(2. - scaling_alpha_), right);
  return true;
}

// AveragePreconditioners on segments: a prox without diagsteps whose range lies inside ONE segment
// averages `cnt` copies of the same value in every group (float running sum, then divide -- the
// rounding of that sum is reproduced); anything else needs the element-wise path.
bool Problem::average_segments(std::vector<ScaleSeg>& segs, const ProxList& prox) {
  for (auto& p : prox) {
    if (p->diagsteps() || p->size() == 0) continue;
    const size_t cnt = p->uniform_group_size();
    if (cnt == 0) return false;
    const size_t lo = p->index(), hi = lo + p->size();
    size_t k = 0;
    while (k < segs.size() && !(segs[k].begin <= lo && lo < segs[k].end)) ++k;
    if (k == segs.size() || hi > segs[k].end) return false;
    const float v = segs[k].value;
    float avg = 0;
    for (size_t c = 0; c < cnt; ++c) avg += v;
    avg /= static_cast<float>(cnt);
    if (avg == v) continue;
    const ScaleSeg old = segs[k];
    std::vector<ScaleSeg> repl;
    if (old.begin < lo) repl.push_back({old.begin, lo, v});
    repl.push_back({lo, hi, avg});
    if (hi < old.end) repl.push_back({hi, old.end, v});
    segs.erase(segs.begin() + k);
    segs.insert(segs.begin() + k, repl.begin(), repl.end());
  }
  return true;
}

static bool is_uniform(const std::vector<float>& v) {
  for (size_t i = 1; i < v.size(); ++i)
    if (v[i] != v[0]) return false;
  return true;
}

void Problem::initialize() {
  ctx_->bind();
  PB_TRACE_SCOPE("Problem::initialize");
  linop_->initialize();
  if (!dims_set_) {
    nrows_ = linop_->nrows();
    ncols_ = linop_->ncols();
  }
  if (linop_->nrows() > nrows_ || linop_->ncols() > ncols_)
    fail(PB_ERR_INVALID, "Size of linear operator exceeds the size of the variables.");
  if (linop_->nrows() != nrows_ || linop_->ncols() != ncols_)
    std::cout << "Size of linear operator (ncols=" << linop_->ncols() << ", nrows=" << linop_->nrows()
              << ") doesn't match size of variables. There might be some unnecessary variables in the problem.\n";
  if (nrows_ >= (1ull << 31) || ncols_ >= (1ull << 31))
    fail(PB_ERR_UNSUPPORTED, "problem dimensions exceed 2^31-1");

  if (prox_f_.empty() && prox_fstar_.empty())
    fail(PB_ERR_INVALID, "No proximal operator for f or fstar specified.");
  if (prox_g_.empty() && prox_gstar_.empty())
    fail(PB_ERR_INVALID, "No proximal operator for g or gstar specified.");
  if (!prox_f_.empty() && !prox_fstar_.empty())
    fail(PB_ERR_INVALID, "Proximal operator for f AND fstar specified. Only set one!");
  if (!prox_g_.empty() && !prox_gstar_.empty())
    fail(PB_ERR_INVALID, "Proximal operator for g AND gstar specified. Only set one!");

  add_zero_prox(ctx_, prox_f_, nrows_, "prox_f");
  add_zero_prox(ctx_, prox_g_, ncols_, "prox_g");
  add_zero_prox(ctx_, prox_fstar_, nrows_, "prox_fstar");
  add_zero_prox(ctx_, prox_gstar_, ncols_, "prox_gstar");
  check_domain_prox(prox_g_, ncols_, "prox_g");
  check_domain_prox(prox_f_, nrows_, "prox_f");
  check_domain_prox(prox_gstar_, ncols_, "prox_gstar");
  check_domain_prox(prox_fstar_, nrows_, "prox_fstar");

  const ProxList& avg_right = prox_g_.empty() ? prox_gstar_ : prox_g_;
  const ProxList& avg_left = prox_f_.empty() ? prox_fstar_ : prox_f_;
  bool done = false;
  {
    // piecewise-constant preconditioners (gradient / zero blocks, identity scaling): a handful of
    // segments instead of nrows + ncols element-wise evaluations, nothing to upload when uniform
    PB_TRACE_SCOPE("Problem::initialize scaling (segments)");
    std::vector<ScaleSeg> ls, rs;
    bool ok = false;
    if (scaling_type_ == kScalingIdentity) {
      ls.push_back({0, nrows_, 1.f});
      rs.push_back({0, ncols_, 1.f});
      ok = true;
    } else if (scaling_type_ == kScalingAlpha) {
      ok = scaling_segments(ls, rs);
    }
    if (ok && average_segments(rs, avg_right) && average_segments(ls, avg_left)) {
      left_.set_segments(nrows_, std::move(ls));
      right_.set_segments(ncols_, std::move(rs));
      done = true;
    }
  }
  if (!done) {
    PB_TRACE_SCOPE("Problem::initialize scaling (element-wise)");
    std::vector<float> left_host, right_host;
    if (scaling_type_ == kScalingAlpha) {
      // Pock-Chambolle: Sigma_r = 1 / sum_c |K_rc|^alpha, T_c = 1 / sum_r |K_rc|^(2-alpha).
      // An empty row/column reuses the previous value, and the carry runs from the last row
      // into the first column because the reference uses one variable (problem.cu:262-287).
      std::vector<float> rs, cs;
      linop_->row_sums(scaling_alpha_, rs);
      linop_->col_sums(static_cast<float>(2. - scaling_alpha_), cs);
      left_host.assign(nrows_, 0.f);
      right_host.assign(ncols_, 0.f);
      float value = 1;
      for (size_t r = 0; r < nrows_; ++r) {
        const float s = r < rs.size() ? rs[r] : 0.f;
        if (s > 0) value = static_cast<float>(1. / s);
        left_host[r] = value;
      }
      for (size_t c = 0; c < ncols_; ++c) {
        const float s = c < cs.size() ? cs[c] : 0.f;
        if (s > 0) value = static_cast<float>(1. / s);
        right_host[c] = value;
      }
    } else if (scaling_type_ == kScalingIdentity) {
      left_host.assign(nrows_, 1.f);
      right_host.assign(ncols_, 1.f);
    } else {
      if (custom_left_.size() != nrows_ || custom_right_.size() != ncols_)
        fail(PB_ERR_INVALID,
             "Preconditioners/diagonal scaling vectors do not fit the size of linear operator.");
      left_host = custom_left_;
      right_host = custom_right_;
    }
    average_preconditioners(right_host, avg_right);
    average_preconditioners(left_host, avg_left);
    left_.set_host(std::move(left_host));
    right_.set_host(std::move(right_host));
  }
  dualized_ = false;
  initialized_ = true;
}

// The element-wise alpha scaling of initialize() for the whole row-sharded operator.  Row sums are complete on
// the rank that owns the row; column sums are this rank's partial sums, added over the ranks in double and
// rounded once.  The carry of the reference (one variable through all rows, then all columns) crosses the ranks:
// rank r's first empty rows take the value of the last non-empty row of ranks < r, and column 0's carry is the
// value of the globally last non-empty row (1 where there is none).
void Problem::shard_alpha_scaling(Comm& comm) {
  ctx_->bind();
  PB_TRACE_SCOPE("Problem::shard_alpha_scaling");
  const int world = comm.world(), rank = comm.rank();
  std::vector<float> rs, cs;
  linop_->row_sums(scaling_alpha_, rs);
  linop_->col_sums(static_cast<float>(2. - scaling_alpha_), cs);
  auto row_sum = [&](size_t r) { return r < rs.size() ? rs[r] : 0.f; };

  // (has a non-empty row, value of the last one) of every rank, in rank order
  std::vector<double> last(2 * (size_t)world + ncols_, 0.0);
  for (size_t r = nrows_; r-- > 0;) {
    const float s = row_sum(r);
    if (s > 0) {
      last[2 * rank] = 1.0;
      last[2 * rank + 1] = static_cast<float>(1. / s);
      break;
    }
  }
  double* col = last.data() + 2 * world;
  for (size_t c = 0; c < cs.size() && c < ncols_; ++c) col[c] = cs[c];
  comm.allreduce_sum_host(last.data(), last.size());

  float value = 1;
  for (int k = 0; k < rank; ++k)
    if (last[2 * k] != 0.0) value = static_cast<float>(last[2 * k + 1]);
  std::vector<float> left_host(nrows_), right_host(ncols_);
  for (size_t r = 0; r < nrows_; ++r) {
    const float s = row_sum(r);
    if (s > 0) value = static_cast<float>(1. / s);
    left_host[r] = value;
  }
  for (int k = rank + 1; k < world; ++k)
    if (last[2 * k] != 0.0) value = static_cast<float>(last[2 * k + 1]);
  for (size_t c = 0; c < ncols_; ++c) {
    const float s = static_cast<float>(col[c]);
    if (s > 0) value = static_cast<float>(1. / s);
    right_host[c] = value;
  }
  average_preconditioners(right_host, prox_g_.empty() ? prox_gstar_ : prox_g_);
  average_preconditioners(left_host, prox_f_.empty() ? prox_fstar_ : prox_f_);
  left_.set_host(std::move(left_host));
  right_.set_host(std::move(right_host));
}

// AveragePreconditioners (problem.cu:502-536): float running sum in group order, then divide.
void Problem::average_preconditioners(std::vector<float>& precond, const ProxList& prox) {
  std::vector<std::tuple<size_t, size_t, size_t>> groups;
  for (auto& p : prox) {
    if (p->diagsteps()) continue;
    // constant preconditioner over the prox' range and equally sized groups (gradient operators):
    // every group averages the same `cnt` copies of one value -- evaluate that float running sum
    // once instead of enumerating millions of groups
    const size_t cnt_u = p->uniform_group_size();
    if (cnt_u > 0 && p->size() > 0 && p->index() + p->size() <= precond.size()) {
      const float* v = precond.data() + p->index();
      bool uniform = true;
      for (size_t i = 1; i < p->size() && uniform; ++i) uniform = v[i] == v[0];
      if (uniform) {
        float avg = 0;
        for (size_t c = 0; c < cnt_u; ++c) avg += v[0];
        avg /= static_cast<float>(cnt_u);
        if (avg != v[0]) std::fill(precond.begin() + p->index(), precond.begin() + p->index() + p->size(), avg);
        continue;
      }
    }
    groups.clear();
    p->get_separable_structure(groups);
    for (auto& g : groups) {
      const size_t idx = std::get<0>(g), cnt = std::get<1>(g), str = std::get<2>(g);
      float avg = 0;
      for (size_t c = 0; c < cnt; ++c) avg += precond[idx + c * str];
      avg /= static_cast<float>(cnt);
      for (size_t c = 0; c < cnt; ++c) precond[idx + c * str] = avg;
    }
  }
}

void Problem::dualize() {
  prox_g_.swap(prox_fstar_);
  prox_gstar_.swap(prox_f_);
  std::swap(nrows_, ncols_);
  left_.swap(right_);
  dualized_ = !dualized_;
}

void Problem::apply_K(float* d_res, const float* d_rhs, bool adjoint) {
  const bool transpose = dualized_ ? !adjoint : adjoint;
  if (!dualized_) linop_->eval(d_res, d_rhs, 0.f, adjoint);
  else linop_->eval(d_res, d_rhs, 0.f, !adjoint, /*negate=*/true);   // dual operator is -K^T
  // variables beyond the operator's extent (SetDimensions larger than the blocks) see K = 0: the
  // reference zero-fills the whole result vector (linearoperator.cu:140-141)
  const size_t covered = transpose ? linop_->ncols() : linop_->nrows();
  const size_t total = adjoint ? ncols_ : nrows_;
  if (total > covered)
    PB_CUDA(cudaMemsetAsync(d_res + covered, 0, (total - covered) * sizeof(float), ctx_->stream));
}

size_t Problem::gpu_mem_amount() const {
  size_t mem = 0;
  for (auto& p : prox_f_) mem += p->gpu_mem_amount();
  for (auto& p : prox_g_) mem += p->gpu_mem_amount();
  for (auto& p : prox_fstar_) mem += p->gpu_mem_amount();
  for (auto& p : prox_gstar_) mem += p->gpu_mem_amount();
  mem += linop_->gpu_mem_amount();
  mem += sizeof(float) * (nrows_ + ncols_);
  return mem;
}

// Power iteration on Sigma^1/2 K T^1/2 (problem.cu:428-500).  `ops` supplies K / K^T and the sum over ranks of
// the two sums of squares of every step (slabs, pb_pdhg.cu); by default the problem's own operator on one GPU.
// The norms are taken from the summed doubles, so every rank sees the same values and stops at the same step.
float Problem::normest(float tol, int max_iters, const float* h_x0, const NormestOps& ops) {
  ctx_->bind();
  const size_t n = ncols_, m = nrows_;
  DeviceBuffer<float> x(n), Ax(m), x_temp(n), Ax_temp(m);
  DeviceBuffer<double> scratch;
  std::vector<float> x_host(n);
  if (h_x0) {
    std::copy(h_x0, h_x0 + n, x_host.begin());
  } else {
    std::srand(0);   // the reference does not seed; a fixed seed keeps runs reproducible
    for (auto& v : x_host) v = (float)std::rand() / (float)RAND_MAX;
  }
  x.upload(x_host.data(), n, ctx_->stream);
  auto sgrid = [&](size_t k) { return (unsigned)std::min<size_t>(grid_for(k), (size_t)ctx_->num_sms * 32); };
  auto apply = [&](float* res, const float* rhs, bool adjoint) {
    if (ops.apply) ops.apply(res, rhs, adjoint);
    else apply_K(res, rhs, adjoint);
  };

  float norm = 0, norm_prev;
  for (int i = 0; i < max_iters; ++i) {
    norm_prev = norm;
    double sq[2];
    mul_sqrt_kernel<<<sgrid(n), kBlock, 0, ctx_->stream>>>(x_temp.data(), scaling_right(), x.data(), n);
    apply(Ax_temp.data(), x_temp.data(), false);
    mul_sqrt_kernel<<<sgrid(m), kBlock, 0, ctx_->stream>>>(Ax.data(), scaling_left(), Ax_temp.data(), m);
    sq[0] = device_sumsq(ctx_, Ax.data(), m, scratch);
    mul_sqrt_kernel<<<sgrid(m), kBlock, 0, ctx_->stream>>>(Ax_temp.data(), scaling_left(), Ax.data(), m);
    apply(x_temp.data(), Ax_temp.data(), true);
    mul_sqrt_kernel<<<sgrid(n), kBlock, 0, ctx_->stream>>>(x.data(), scaling_right(), x_temp.data(), n);
    PB_CHECK_LAUNCH();
    ctx_->launches += 4;
    sq[1] = device_sumsq(ctx_, x.data(), n, scratch);
    if (ops.sum) ops.sum(sq, 2);
    const float norm_Ax = std::sqrt(static_cast<float>(sq[0]));
    const float norm_x = std::sqrt(static_cast<float>(sq[1]));
    norm = norm_x / norm_Ax;
    if (std::abs(norm_prev - norm) < tol * norm) break;
    divide_kernel<<<sgrid(n), kBlock, 0, ctx_->stream>>>(x.data(), n, norm_x);
    PB_CHECK_LAUNCH();
    ctx_->launches++;
  }
  return norm;
}

}  // namespace pb
