// pb_capi.cu -- extern "C" boundary (include/prost_b200.h) and the Solver loop
// (Solver<T>::Solve, src/solver.cu:122-209).
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <thread>
#include <iomanip>
#include <iostream>
#include <new>

#include "pb_backend.cuh"

namespace pb { unsigned tile_ring_trace_read(unsigned long long* h_out, unsigned n); }   // pb_tile.cu
#include "pb_comm.cuh"
#include "pb_problem.cuh"

#ifndef PB_VERSION
#define PB_VERSION "prost-b200 0.1"
#endif

struct pb_context { pb::Context ctx; };
struct pb_block { std::shared_ptr<pb::Block> impl; };
struct pb_linop { pb::Context* ctx; std::shared_ptr<pb::LinearOperator> impl; bool initialized = false; };
struct pb_prox { pb::Context* ctx; std::shared_ptr<pb::Prox> impl; };
struct pb_problem { std::shared_ptr<pb::Problem> impl; };
struct pb_backend { std::shared_ptr<pb::Backend> impl; };
struct pb_comm { std::unique_ptr<pb::Comm> impl; };

namespace {

thread_local std::string g_last_error;

int set_error(int status, const std::string& msg) {
  g_last_error = msg;
  return status;
}

template <typename F>
int guarded(F&& f) {
  try {
    f();
    return PB_OK;
  } catch (const pb::Error& e) {
    return set_error(e.status, e.what());
  } catch (const std::bad_alloc& e) {
    return set_error(PB_ERR_OOM, std::string("Out of memory: ") + e.what());
  } catch (const std::exception& e) {
    return set_error(PB_ERR_INVALID, e.what());
  }
}

void require(bool cond, const char* msg) {
  if (!cond) pb::fail(PB_ERR_INVALID, msg);
}

}  // namespace

extern "C" {

const char* pb_version(void) { return PB_VERSION; }
const char* pb_last_error(void) { return g_last_error.c_str(); }

int pb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int pb_context_create(int device, void* stream, pb_context** out) {
  return guarded([&] {
    require(out != nullptr, "pb_context_create: out is NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
      cudaGetLastError();
      pb::fail(PB_ERR_CUDA, std::string("CUDA error: no usable CUDA device (") +
                                (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                                "); prost_b200 has no CPU fallback");
    }
    require(device >= 0 && device < n, "pb_context_create: device index out of range");
    auto* c = new pb_context();
    c->ctx.device = device;
    PB_CUDA(cudaSetDevice(device));
    if (stream) {
      c->ctx.stream = static_cast<cudaStream_t>(stream);
      c->ctx.owns_stream = false;
    } else {
      PB_CUDA(cudaStreamCreateWithFlags(&c->ctx.stream, cudaStreamNonBlocking));
      c->ctx.owns_stream = true;
    }
    int sms = 0;
    PB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    c->ctx.num_sms = sms > 0 ? sms : pb::kNumSMs;
    *out = c;
  });
}

void pb_context_destroy(pb_context* c) {
  if (!c) return;
  cudaSetDevice(c->ctx.device);
  pb::release_host_staging(&c->ctx);
  if (c->ctx.owns_stream && c->ctx.stream) cudaStreamDestroy(c->ctx.stream);
  delete c;
}

void pb_release_cached_memory(void) { pb::device_cache_release(); }

int pb_context_synchronize(pb_context* c) {
  return guarded([&] {
    require(c != nullptr, "NULL context");
    c->ctx.bind();
    PB_CUDA(cudaStreamSynchronize(c->ctx.stream));
  });
}
void* pb_context_stream(pb_context* c) { return c ? static_cast<void*>(c->ctx.stream) : nullptr; }
int pb_context_device(pb_context* c) { return c ? c->ctx.device : -1; }

int pb_host_alloc(size_t bytes, void** h_out) {
  return guarded([&] { require(h_out != nullptr, "pb_host_alloc: NULL argument"); *h_out = pb::host_pool_alloc(bytes); });
}
void pb_host_free(void* p) { pb::host_pool_free(p); }
int pb_malloc(pb_context* c, size_t bytes, void** d_out) {
  return guarded([&] {
    require(c && d_out, "pb_malloc: NULL argument");
    c->ctx.bind();
    PB_CUDA(cudaMalloc(d_out, bytes));
  });
}
int pb_free(pb_context* c, void* p) {
  return guarded([&] {
    require(c != nullptr, "NULL context");
    c->ctx.bind();
    PB_CUDA(cudaFree(p));
  });
}
int pb_memcpy_h2d(pb_context* c, void* d, const void* h, size_t bytes) {
  return guarded([&] {
    require(c != nullptr, "NULL context");
    c->ctx.bind();
    PB_CUDA(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, c->ctx.stream));
    PB_CUDA(cudaStreamSynchronize(c->ctx.stream));
  });
}
int pb_memcpy_d2h(pb_context* c, void* h, const void* d, size_t bytes) {
  return guarded([&] {
    require(c != nullptr, "NULL context");
    c->ctx.bind();
    PB_CUDA(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, c->ctx.stream));
    PB_CUDA(cudaStreamSynchronize(c->ctx.stream));
  });
}

// ---- blocks --------------------------------------------------------------------------------------

#define PB_MAKE_BLOCK(expr)                                  \
  return guarded([&] {                                       \
    require(c && out, "block create: NULL argument");        \
    c->ctx.bind();                                           \
    auto* h = new pb_block();                                \
    try { h->impl = (expr); } catch (...) { delete h; throw; } \
    *out = h;                                                \
  })

int pb_block_create_gradient2d(pb_context* c, size_t row, size_t col, size_t nx, size_t ny, size_t L,
                               int label_first, pb_block** out) {
  PB_MAKE_BLOCK(pb::make_block_gradient(&c->ctx, false, row, col, nx, ny, L, label_first != 0));
}
int pb_block_create_gradient3d(pb_context* c, size_t row, size_t col, size_t nx, size_t ny, size_t L,
                               int label_first, pb_block** out) {
  PB_MAKE_BLOCK(pb::make_block_gradient(&c->ctx, true, row, col, nx, ny, L, label_first != 0));
}
int pb_block_create_diags(pb_context* c, size_t row, size_t col, size_t nrows, size_t ncols,
                          size_t ndiags, const int64_t* offsets, const float* factors, pb_block** out) {
  PB_MAKE_BLOCK(pb::make_block_diags(&c->ctx, row, col, nrows, ncols, ndiags, offsets, factors));
}
int pb_block_create_sparse_csc(pb_context* c, size_t row, size_t col, int m, int n, int nnz,
                               const float* val, const int32_t* ptr, const int32_t* ind, pb_block** out) {
  PB_MAKE_BLOCK(pb::make_block_sparse_csc(&c->ctx, row, col, m, n, nnz, val, ptr, ind));
}
int pb_block_create_dense(pb_context* c, size_t row, size_t col, size_t nrows, size_t ncols,
                          const float* data, pb_block** out) {
  PB_MAKE_BLOCK(pb::make_block_dense(&c->ctx, row, col, nrows, ncols, data));
}
int pb_block_create_dense_kron_id(pb_context* c, size_t diaglength, size_t row, size_t col, size_t nrows,
                                  size_t ncols, const float* data, pb_block** out) {
  PB_MAKE_BLOCK(pb::make_block_dense_kron(&c->ctx, false, diaglength, row, col, nrows, ncols, data));
}
int pb_block_create_id_kron_dense(pb_context* c, size_t diaglength, size_t row, size_t col, size_t nrows,
                                  size_t ncols, const float* data, pb_block** out) {
  PB_MAKE_BLOCK(pb::make_block_dense_kron(&c->ctx, true, diaglength, row, col, nrows, ncols, data));
}
int pb_block_create_sparse_kron_id(pb_context* c, size_t row, size_t col, size_t diaglength, int m, int n, int nnz,
                                   const float* val, const int32_t* ptr, const int32_t* ind, pb_block** out) {
  PB_MAKE_BLOCK((require(val && ptr && ind, "NULL argument"),
                 pb::make_block_sparse_kron(&c->ctx, false, diaglength, row, col, m, n, nnz, val, ptr, ind)));
}
int pb_block_create_id_kron_sparse(pb_context* c, size_t row, size_t col, size_t diaglength, int m, int n, int nnz,
                                   const float* val, const int32_t* ptr, const int32_t* ind, pb_block** out) {
  PB_MAKE_BLOCK((require(val && ptr && ind, "NULL argument"),
                 pb::make_block_sparse_kron(&c->ctx, true, diaglength, row, col, m, n, nnz, val, ptr, ind)));
}
int pb_block_create_zero(pb_context* c, size_t row, size_t col, size_t nrows, size_t ncols,
                         pb_block** out) {
  PB_MAKE_BLOCK(pb::make_block_zero(&c->ctx, row, col, nrows, ncols));
}
void pb_block_destroy(pb_block* b) { delete b; }
size_t pb_block_row(const pb_block* b) { return b->impl->row(); }
size_t pb_block_col(const pb_block* b) { return b->impl->col(); }
size_t pb_block_nrows(const pb_block* b) { return b->impl->nrows(); }
size_t pb_block_ncols(const pb_block* b) { return b->impl->ncols(); }
float pb_block_row_sum(const pb_block* b, size_t row, float alpha) { return b->impl->row_sum(row, alpha); }
float pb_block_col_sum(const pb_block* b, size_t col, float alpha) { return b->impl->col_sum(col, alpha); }
size_t pb_block_gpu_mem_amount(const pb_block* b) { return b->impl->gpu_mem_amount(); }

// ---- linear operator ---------------------------------------------------------------------------

int pb_linop_create(pb_context* c, pb_linop** out) {
  return guarded([&] {
    require(c && out, "pb_linop_create: NULL argument");
    auto* h = new pb_linop();
    h->ctx = &c->ctx;
    h->impl = std::make_shared<pb::LinearOperator>(&c->ctx);
    *out = h;
  });
}
void pb_linop_destroy(pb_linop* op) { delete op; }
int pb_linop_add_block(pb_linop* op, pb_block* b) {
  return guarded([&] {
    require(op && b, "pb_linop_add_block: NULL argument");
    op->impl->add_block(b->impl);
  });
}
int pb_linop_initialize(pb_linop* op) {
  return guarded([&] {
    require(op != nullptr, "NULL linop");
    op->impl->initialize();
    op->initialized = true;
  });
}
size_t pb_linop_nrows(const pb_linop* op) { return op->impl->nrows(); }
size_t pb_linop_ncols(const pb_linop* op) { return op->impl->ncols(); }
int pb_linop_eval(pb_linop* op, float* d_result, const float* d_rhs, float beta, int transpose) {
  return guarded([&] {
    require(op && op->initialized, "LinearOperator has not been initialized.");
    op->impl->eval(d_result, d_rhs, beta, transpose != 0);
  });
}
int pb_linop_eval_host(pb_linop* op, float* h_result, const float* h_rhs, int transpose, double* ms_out) {
  return guarded([&] {
    require(op && op->initialized, "LinearOperator has not been initialized.");
    pb::Context* ctx = op->ctx;
    ctx->bind();
    const size_t nin = transpose ? op->impl->nrows() : op->impl->ncols();
    const size_t nout = transpose ? op->impl->ncols() : op->impl->nrows();
    pb::DeviceBuffer<float> d_in(nin), d_out(nout);
    d_in.upload(h_rhs, nin, ctx->stream);
    cudaEvent_t e0, e1;
    PB_CUDA(cudaEventCreate(&e0));
    PB_CUDA(cudaEventCreate(&e1));
    const int repeats = 5;                       // linearoperator.cu:177
    PB_CUDA(cudaEventRecord(e0, ctx->stream));
    for (int i = 0; i < repeats; ++i) op->impl->eval(d_out.data(), d_in.data(), 0.f, transpose != 0);
    PB_CUDA(cudaEventRecord(e1, ctx->stream));
    PB_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    PB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    d_out.download(h_result, nout, ctx->stream);
    PB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (ms_out) *ms_out = ms / repeats;
  });
}
float pb_linop_row_sum(const pb_linop* op, size_t row, float alpha) { return op->impl->row_sum(row, alpha); }
float pb_linop_col_sum(const pb_linop* op, size_t col, float alpha) { return op->impl->col_sum(col, alpha); }
int pb_linop_row_sums(const pb_linop* op, float alpha, float* h_out) {
  return guarded([&] {
    std::vector<float> v;
    op->impl->row_sums(alpha, v);
    std::copy(v.begin(), v.end(), h_out);
  });
}
int pb_linop_col_sums(const pb_linop* op, float alpha, float* h_out) {
  return guarded([&] {
    std::vector<float> v;
    op->impl->col_sums(alpha, v);
    std::copy(v.begin(), v.end(), h_out);
  });
}

// ---- prox ----------------------------------------------------------------------------------------

int pb_function1d_from_name(const char* name) {
  // names of the mex registry (factory.cpp:20-47: "elem_operation:1d:<name>")
  static const char* names[] = {"zero", "abs", "square", "ind_leq0", "ind_geq0", "ind_eq0", "ind_box01",
                                "max_pos0", "l0", "huber", "lq", "lq_plus_eps", "truncquad", "trunclin"};
  if (!name) return -1;
  for (int i = 0; i < PB_FUN_COUNT_; ++i)
    if (std::strcmp(name, names[i]) == 0) return i;
  if (std::strcmp(name, "trunc_quad") == 0) return PB_FUN_TRUNC_QUAD;
  if (std::strcmp(name, "trunc_linear") == 0) return PB_FUN_TRUNC_LINEAR;
  return -1;
}

#define PB_MAKE_PROX(expr)                                     \
  return guarded([&] {                                         \
    require(c && out, "prox create: NULL argument");           \
    c->ctx.bind();                                             \
    auto* h = new pb_prox();                                   \
    h->ctx = &c->ctx;                                          \
    try { h->impl = (expr); } catch (...) { delete h; throw; } \
    *out = h;                                                  \
  })

int pb_prox_create_elem_1d(pb_context* c, size_t index, size_t count, size_t dim, int interleaved,
                           int diagsteps, int function, const float* const coeffs[7],
                           const size_t coeff_len[7], pb_prox** out) {
  PB_MAKE_PROX(pb::make_prox_elem(&c->ctx, pb::kProxElem1D, index, count, dim, interleaved != 0,
                                  diagsteps != 0, function, coeffs, coeff_len));
}
int pb_prox_create_elem_norm2(pb_context* c, size_t index, size_t count, size_t dim, int interleaved,
                              int diagsteps, int function, const float* const coeffs[7],
                              const size_t coeff_len[7], pb_prox** out) {
  PB_MAKE_PROX(pb::make_prox_elem(&c->ctx, pb::kProxNorm2, index, count, dim, interleaved != 0,
                                  diagsteps != 0, function, coeffs, coeff_len));
}
int pb_prox_create_ind_simplex(pb_context* c, size_t index, size_t count, size_t dim, int interleaved,
                               int diagsteps, pb_prox** out) {
  PB_MAKE_PROX(pb::make_prox_simplex(&c->ctx, index, count, dim, interleaved != 0, diagsteps != 0));
}
int pb_prox_create_ind_sum(pb_context* c, size_t index, size_t count, size_t dim, int interleaved, int diagsteps,
                           pb_prox** out) {
  PB_MAKE_PROX(pb::make_prox_ind_sum(&c->ctx, index, count, dim, interleaved != 0, diagsteps != 0));
}
int pb_prox_create_ind_sum_indexed(pb_context* c, size_t index, size_t size, size_t count, size_t dim,
                                   const unsigned long long* inds, float sum, size_t count2, size_t dim2,
                                   const unsigned long long* inds2, float sum2, pb_prox** out) {
  PB_MAKE_PROX(pb::make_prox_ind_sum_indexed(&c->ctx, index, size, count, dim, inds, sum, count2, dim2, inds2, sum2));
}
int pb_prox_create_spectral(pb_context* c, int kind, size_t index, size_t count, size_t dim, int interleaved,
                            int diagsteps, int function_1d, int function_2d, const float* const coeffs[7],
                            const size_t coeff_len[7], pb_prox** out) {
  PB_MAKE_PROX((require(coeffs && coeff_len, "NULL coefficients"),
                pb::make_prox_spectral(&c->ctx, kind, index, count, dim, interleaved != 0, diagsteps != 0, function_1d,
                                       function_2d, coeffs, coeff_len)));
}
int pb_prox_create_ind_range(pb_context* c, size_t index, size_t size, int diagsteps, int m, int n, int nnz,
                             const float* val, const int32_t* ptr, const int32_t* ind, const float* aa, pb_prox** out) {
  PB_MAKE_PROX(pb::make_prox_ind_range(&c->ctx, index, size, diagsteps != 0, m, n, nnz, val, ptr, ind, aa));
}
int pb_prox_create_ind_epi_conjquad_1d(pb_context* c, size_t index, size_t count, int interleaved, int diagsteps,
                                       const float* const coeffs[5], const size_t coeff_len[5], pb_prox** out) {
  PB_MAKE_PROX((require(coeffs && coeff_len, "NULL coefficients"),
                pb::make_prox_ind_epi_conjquad_1d(&c->ctx, index, count, interleaved != 0, diagsteps != 0, coeffs, coeff_len)));
}
int pb_prox_create_ind_halfspace(pb_context* c, size_t index, size_t count, size_t dim, int interleaved, int diagsteps,
                                 const float* a, size_t na, const float* b, size_t nb, pb_prox** out) {
  PB_MAKE_PROX(pb::make_prox_ind_halfspace(&c->ctx, index, count, dim, interleaved != 0, diagsteps != 0, a, na, b, nb));
}
int pb_prox_create_ind_soc(pb_context* c, size_t index, size_t count, size_t dim, int interleaved, int diagsteps,
                           float alpha, pb_prox** out) {
  PB_MAKE_PROX(pb::make_prox_ind_soc(&c->ctx, index, count, dim, interleaved != 0, diagsteps != 0, alpha));
}
int pb_prox_create_ind_epi_quad(pb_context* c, size_t index, size_t count, size_t dim, int interleaved,
                                int diagsteps, const float* a, size_t na, const float* b, size_t nb,
                                const float* cc, size_t nc, pb_prox** out) {
  PB_MAKE_PROX(pb::make_prox_epi_quad(&c->ctx, index, count, dim, interleaved != 0, diagsteps != 0, a, na,
                                      b, nb, cc, nc));
}
int pb_prox_create_moreau(pb_context* c, pb_prox* conjugate, pb_prox** out) {
  PB_MAKE_PROX((require(conjugate != nullptr, "NULL prox"), pb::make_prox_moreau(&c->ctx, conjugate->impl)));
}
int pb_prox_create_permute(pb_context* c, pb_prox* base, const int* perm, size_t n, pb_prox** out) {
  PB_MAKE_PROX((require(base != nullptr, "NULL prox"), pb::make_prox_permute(&c->ctx, base->impl, perm, n)));
}
int pb_prox_create_transform(pb_context* c, pb_prox* inner, const float* const coeffs[5], const size_t coeff_len[5],
                             pb_prox** out) {
  PB_MAKE_PROX((require(inner != nullptr && coeffs != nullptr && coeff_len != nullptr, "NULL argument"),
                pb::make_prox_transform(&c->ctx, inner->impl, coeffs, coeff_len)));
}
int pb_prox_create_zero(pb_context* c, size_t index, size_t size, pb_prox** out) {
  PB_MAKE_PROX(pb::make_prox_zero(&c->ctx, index, size));
}
void pb_prox_destroy(pb_prox* p) { delete p; }
size_t pb_prox_index(const pb_prox* p) { return p->impl->index(); }
size_t pb_prox_size(const pb_prox* p) { return p->impl->size(); }
int pb_prox_diagsteps(const pb_prox* p) { return p->impl->diagsteps() ? 1 : 0; }
size_t pb_prox_gpu_mem_amount(const pb_prox* p) { return p->impl->gpu_mem_amount(); }

int pb_prox_eval(pb_prox* p, float* d_result, const float* d_arg, const float* d_tau_diag, float tau,
                 int invert_tau) {
  return guarded([&] {
    require(p != nullptr, "NULL prox");
    p->impl->eval(d_result, d_arg, d_tau_diag, tau, invert_tau != 0);
  });
}

int pb_prox_eval_host(pb_prox* p, float* h_result, const float* h_arg, const float* h_tau_diag, size_t n,
                      float tau, int invert_tau, double* ms_out) {
  return guarded([&] {
    require(p != nullptr, "NULL prox");
    require(p->impl->index() + p->impl->size() <= n, "pb_prox_eval_host: vectors shorter than the prox range");
    pb::Context* ctx = p->ctx;
    ctx->bind();
    pb::DeviceBuffer<float> d_arg(n), d_res(n), d_tau(n);
    d_arg.upload(h_arg, n, ctx->stream);
    d_tau.upload(h_tau_diag, n, ctx->stream);
    d_res.zero(ctx->stream);
    cudaEvent_t e0, e1;
    PB_CUDA(cudaEventCreate(&e0));
    PB_CUDA(cudaEventCreate(&e1));
    PB_CUDA(cudaEventRecord(e0, ctx->stream));
    p->impl->eval(d_res.data(), d_arg.data(), d_tau.data(), tau, invert_tau != 0);
    PB_CUDA(cudaEventRecord(e1, ctx->stream));
    PB_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    PB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    d_res.download(h_result, n, ctx->stream);
    PB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (ms_out) *ms_out = ms;
  });
}

// ---- problem -------------------------------------------------------------------------------------

int pb_problem_create(pb_context* c, pb_problem** out) {
  return guarded([&] {
    require(c && out, "pb_problem_create: NULL argument");
    auto* h = new pb_problem();
    h->impl = std::make_shared<pb::Problem>(&c->ctx);
    *out = h;
  });
}
void pb_problem_destroy(pb_problem* p) { delete p; }
int pb_problem_add_block(pb_problem* p, pb_block* b) {
  return guarded([&] { require(p && b, "NULL argument"); p->impl->add_block(b->impl); });
}
int pb_problem_add_prox_g(pb_problem* p, pb_prox* x) {
  return guarded([&] { require(p && x, "NULL argument"); p->impl->add_prox_g(x->impl); });
}
int pb_problem_add_prox_f(pb_problem* p, pb_prox* x) {
  return guarded([&] { require(p && x, "NULL argument"); p->impl->add_prox_f(x->impl); });
}
int pb_problem_add_prox_gstar(pb_problem* p, pb_prox* x) {
  return guarded([&] { require(p && x, "NULL argument"); p->impl->add_prox_gstar(x->impl); });
}
int pb_problem_add_prox_fstar(pb_problem* p, pb_prox* x) {
  return guarded([&] { require(p && x, "NULL argument"); p->impl->add_prox_fstar(x->impl); });
}
int pb_problem_set_dimensions(pb_problem* p, size_t nrows, size_t ncols) {
  return guarded([&] { require(p != nullptr, "NULL problem"); p->impl->set_dimensions(nrows, ncols); });
}
int pb_problem_set_scaling_alpha(pb_problem* p, float alpha) {
  return guarded([&] { require(p != nullptr, "NULL problem"); p->impl->set_scaling_alpha(alpha); });
}
int pb_problem_set_scaling_identity(pb_problem* p) {
  return guarded([&] { require(p != nullptr, "NULL problem"); p->impl->set_scaling_identity(); });
}
int pb_problem_set_scaling_custom(pb_problem* p, const float* left, size_t nl, const float* right, size_t nr) {
  return guarded([&] { require(p != nullptr, "NULL problem"); p->impl->set_scaling_custom(left, nl, right, nr); });
}
int pb_problem_initialize(pb_problem* p) {
  return guarded([&] { require(p != nullptr, "NULL problem"); p->impl->initialize(); });
}
int pb_problem_dualize(pb_problem* p) {
  return guarded([&] { require(p != nullptr, "NULL problem"); p->impl->dualize(); });
}
size_t pb_problem_nrows(const pb_problem* p) { return p->impl->nrows(); }
size_t pb_problem_ncols(const pb_problem* p) { return p->impl->ncols(); }
size_t pb_problem_gpu_mem_amount(const pb_problem* p) { return p->impl->gpu_mem_amount(); }
int pb_problem_normest(pb_problem* p, float tol, int max_iters, const float* h_x0, float* out) {
  return guarded([&] {
    require(p && out, "NULL argument");
    require(p->impl->initialized(), "Problem has not been initialized.");
    *out = p->impl->normest(tol, max_iters, h_x0);
  });
}
int pb_problem_get_scaling(const pb_problem* p, float* h_left, float* h_right) {
  return guarded([&] {
    require(p != nullptr, "NULL problem");
    const auto& l = p->impl->scaling_left_host();
    const auto& r = p->impl->scaling_right_host();
    if (h_left) std::copy(l.begin(), l.end(), h_left);
    if (h_right) std::copy(r.begin(), r.end(), h_right);
  });
}

// ---- backends ------------------------------------------------------------------------------------

void pb_solver_default_options(pb_solver_options* o) {   // matlab/+prost/options.m:3-14
  o->tol_rel_primal = o->tol_rel_dual = o->tol_abs_primal = o->tol_abs_dual = 1e-4f;
  o->max_iters = 1000;
  o->num_cback_calls = 10;
  o->verbose = 1;
  o->solve_dual_problem = 0;
}
void pb_pdhg_default_options(pb_pdhg_options* o) {       // matlab/+prost/+backend/pdhg.m:3-14
  o->tau0 = 1;
  o->sigma0 = 1;
  o->residual_iter = 1;
  o->scale_steps_operator = 1;
  o->alg2_gamma = 0;
  o->arg_alpha0 = 0.5f;
  o->arg_nu = 0.95f;
  o->arg_delta = 1.5f;
  o->arb_delta = 1.05f;
  o->arb_tau = 0.8f;
  o->stepsize_variant = PB_PDHG_BOYD;
  o->fuse = 1;
  o->normest_x0 = nullptr;
}
void pb_admm_default_options(pb_admm_options* o) {       // matlab/+prost/+backend/admm.m:3-13
  o->rho0 = 1;
  o->alpha = 1.7;
  o->cg_tol_pow = 1.3;
  o->cg_tol_min = 1e-5;
  o->cg_tol_max = 1e-8;
  o->cg_max_iter = 10;
  o->residual_iter = 1;
  o->arb_delta = 1.05f;
  o->arb_tau = 0.8f;
  o->arb_gamma = 1.01f;
}

int pb_pdhg_create(pb_context* c, pb_problem* prob, const pb_pdhg_options* opts,
                   const pb_solver_options* sopts, pb_backend** out) {
  return guarded([&] {
    require(c && prob && opts && sopts && out, "pb_pdhg_create: NULL argument");
    auto* h = new pb_backend();
    try { h->impl = pb::make_backend_pdhg(&c->ctx, prob->impl, *opts, *sopts); } catch (...) { delete h; throw; }
    h->impl->launch_base = c->ctx.launches;
    *out = h;
  });
}
int pb_admm_create(pb_context* c, pb_problem* prob, const pb_admm_options* opts,
                   const pb_solver_options* sopts, pb_backend** out) {
  return guarded([&] {
    require(c && prob && opts && sopts && out, "pb_admm_create: NULL argument");
    auto* h = new pb_backend();
    try { h->impl = pb::make_backend_admm(&c->ctx, prob->impl, *opts, *sopts); } catch (...) { delete h; throw; }
    h->impl->launch_base = c->ctx.launches;
    *out = h;
  });
}
void pb_backend_destroy(pb_backend* b) { delete b; }
int pb_backend_set_solver_options(pb_backend* b, const pb_solver_options* sopts) {
  return guarded([&] { require(b && sopts, "NULL argument"); b->impl->set_solver_options(*sopts); });
}
int pb_backend_initialize(pb_backend* b, const float* h_x0, size_t nx0, const float* h_y0, size_t ny0) {
  return guarded([&] { require(b != nullptr, "NULL backend"); b->impl->initialize(h_x0, nx0, h_y0, ny0); });
}
int pb_backend_iterate(pb_backend* b, int n_iters) {
  return guarded([&] { require(b != nullptr, "NULL backend"); b->impl->iterate(n_iters); });
}
int pb_backend_profile(pb_backend* b, int n_iters, float out_ms[3]) {
  return guarded([&] { require(b && out_ms, "NULL argument"); b->impl->profile(n_iters, out_ms); });
}
int pb_backend_profile_detail(pb_backend* b, int n_iters, float out[8]) {
  return guarded([&] { require(b && out, "NULL argument"); b->impl->profile_detail(n_iters, out); });
}
int pb_backend_residuals(pb_backend* b, float out[6]) {
  return guarded([&] { require(b && out, "NULL argument"); b->impl->residuals(out); });
}
int pb_backend_stepsizes(pb_backend* b, double out[3]) {
  return guarded([&] { require(b && out, "NULL argument"); b->impl->stepsizes(out); });
}
size_t pb_backend_iteration(const pb_backend* b) { return b->impl->iteration(); }
int pb_backend_current_solution(pb_backend* b, float* h_x, float* h_z, float* h_y, float* h_w) {
  return guarded([&] { require(b != nullptr, "NULL backend"); b->impl->current_solution(h_x, h_z, h_y, h_w); });
}
size_t pb_backend_gpu_mem_amount(const pb_backend* b) { return b->impl->gpu_mem_amount(); }
int pb_backend_is_fused(const pb_backend* b) { return b->impl->is_fused() ? 1 : 0; }
unsigned long long pb_backend_one_pass_iterations(const pb_backend* b) { return b->impl->one_pass_iterations(); }
unsigned long long pb_backend_launch_count(const pb_backend* b) {
  return b->impl->ctx()->launches - b->impl->launch_base;
}
int pb_backend_device_iterates(pb_backend* b, float** d_x, float** d_y) {
  return guarded([&] { require(b && d_x && d_y, "NULL argument"); b->impl->device_iterates(d_x, d_y); });
}

unsigned pb_ring_trace_read(unsigned long long* h_out, unsigned n) { return pb::tile_ring_trace_read(h_out, n); }

// ---- slab decomposition --------------------------------------------------------------------------

int pb_comm_unique_id(void* h_id_out) {
  return guarded([&] { require(h_id_out != nullptr, "NULL argument"); pb::Comm::unique_id(h_id_out); });
}
int pb_comm_create(pb_context* c, int rank, int world, const void* h_id, pb_comm** out) {
  return guarded([&] {
    require(c && out, "pb_comm_create: NULL argument");
    auto* h = new pb_comm();
    try { h->impl.reset(new pb::Comm(&c->ctx, rank, world, h_id)); } catch (...) { delete h; throw; }
    *out = h;
  });
}
void pb_comm_destroy(pb_comm* c) { delete c; }
int pb_comm_rank(const pb_comm* c) { return c ? c->impl->rank() : -1; }
int pb_comm_world(const pb_comm* c) { return c ? c->impl->world() : 0; }
int pb_comm_peer_to_peer(const pb_comm* c) { return c && c->impl->p2p() ? 1 : 0; }
int pb_comm_barrier(pb_comm* c) {
  return guarded([&] { require(c != nullptr, "NULL comm"); c->impl->barrier(); });
}
int pb_comm_allreduce_sum(pb_comm* c, double* h_buf, size_t n) {
  return guarded([&] { require(c && h_buf, "NULL argument"); c->impl->allreduce_sum_host(h_buf, n); });
}
int pb_backend_set_slab(pb_backend* b, pb_comm* c) {
  return guarded([&] { require(b && c, "NULL argument"); b->impl->set_slab(c->impl.get()); });
}

// ---- solver loop ---------------------------------------------------------------------------------

int pb_solver_solve(pb_backend* b, const pb_solver_options* so, pb_stopping_cb stop, pb_interm_cb interm,
                    void* user, float* h_x, float* h_z, float* h_y, float* h_w, int* result_out,
                    int* iters_out) {
  return guarded([&] {
    require(b && so, "pb_solver_solve: NULL argument");
    pb::Backend* be = b->impl.get();
    const size_t m = be->problem()->nrows(), n = be->problem()->ncols();
    std::vector<float> x, z, y, w;
    float* px = h_x; float* pz = h_z; float* py = h_y; float* pw = h_w;
    if (!px) { x.resize(n); px = x.data(); }
    if (!py) { y.resize(m); py = y.data(); }
    if (!pz) { z.resize(m); pz = z.data(); }
    if (!pw) { w.resize(n); pw = w.data(); }

    // Fault the (pageable) result buffers in on a helper thread while the GPU iterates: the final
    // read-back of x, z, y, w then lands in resident pages (pb_hostio.cu).  Joined before the first copy.
    std::thread prefault([=] {      // one thread per buffer: short solves must not wait for 400 MB of page faults
      std::thread ty([=] { pb::prefault_host_range(py, m * sizeof(float)); });
      std::thread tz([=] { pb::prefault_host_range(pz, m * sizeof(float)); });
      std::thread tw([=] { pb::prefault_host_range(pw, n * sizeof(float)); });
      pb::prefault_host_range(px, n * sizeof(float));
      ty.join();
      tz.join();
      tw.join();
    });
    struct Joiner {
      std::thread& t;
      ~Joiner() { if (t.joinable()) t.join(); }
    } joiner{prefault};

    // callback schedule: linspace(0, max_iters-1, num_cback_calls) plus the end point
    // (solver.cu:130-135, common.cu:32-46)
    std::deque<double> cb_iters;
    if (so->num_cback_calls >= 2) {
      const double start = 0.0, end = static_cast<double>(so->max_iters - 1);
      const double delta = (end - start) / (static_cast<double>(so->num_cback_calls) - 1.0);
      for (int i = 0; i < so->num_cback_calls; ++i) cb_iters.push_back(start + delta * i);
      cb_iters.push_back(end);
    } else {
      cb_iters.push_back(1e8);
    }

    int result = PB_STOPPED_MAX_ITERS;
    int iters = 0;
    float res[6] = {0, 0, 0, 0, 0, 0};
    for (int i = 0; i < so->max_iters; ++i) {
      const size_t it_before = be->iteration();
      be->iterate(1);
      iters = i + 1;
      // residuals only change on refresh iterations; everything in between reuses the cached
      // values exactly like Solver::Solve does, without synchronising the stream
      if (be->refreshes_on(it_before)) be->residuals(res);
      const bool is_stopped = stop ? stop(user) != 0 : false;
      bool is_converged = (res[0] < res[4]) && (res[1] < res[5]);

      const double front = cb_iters.empty() ? 1e300 : cb_iters.front();
      if (i >= front || is_converged || is_stopped || i == so->max_iters - 1) {
        if (prefault.joinable()) prefault.join();
        be->current_solution(px, pz, py, pw);
        if (so->num_cback_calls >= 1) {
          if (so->verbose) {
            const int digits = static_cast<int>(std::floor(std::log10(static_cast<double>(so->max_iters)))) + 1;
            std::cout << "It " << std::setw(digits) << (i + 1) << ": " << std::scientific
                      << "Feas_p=" << std::setprecision(2) << res[0] << ", Eps_p=" << std::setprecision(2)
                      << res[4] << ", Feas_d=" << std::setprecision(2) << res[1]
                      << ", Eps_d=" << std::setprecision(2) << res[5] << "; " << std::flush;
          }
          if (interm) {
            if (so->solve_dual_problem) is_converged |= interm(user, i + 1, py, m, px, n) != 0;
            else is_converged |= interm(user, i + 1, px, n, py, m) != 0;
          } else if (so->verbose) {
            std::cout << std::endl;
          }
        }
        if (!cb_iters.empty()) cb_iters.pop_front();
      }
      if (is_stopped) {
        if (so->verbose) std::cout << "Stopped by user." << std::endl;
        result = PB_STOPPED_USER;
        break;
      }
      if (is_converged) {
        if (so->verbose) std::cout << "Reached convergence tolerance." << std::endl;
        result = PB_CONVERGED;
        break;
      }
    }
    if (so->verbose && result == PB_STOPPED_MAX_ITERS)
      std::cout << "Reached maximum of " << so->max_iters << " iterations." << std::endl;
    if (prefault.joinable()) prefault.join();
    if (so->max_iters <= 0) be->current_solution(px, pz, py, pw);
    if (result_out) *result_out = result;
    if (iters_out) *iters_out = iters;
  });
}

}  // extern "C"
