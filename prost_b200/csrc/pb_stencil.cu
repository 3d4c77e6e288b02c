// pb_stencil.cu -- pattern matching and launch of the specialised gradient passes (pb_stencil.cuh).
// Compiled once per PB_STENCIL_PART (0..3) so the instantiations build in parallel:
//   part 0  planner + primal kernels with one-element groups (Elem1D / Zero)
//   part 1  primal kernels with per-pixel label groups (simplex)
//   part 2  dual Norm2 kernels on the gradient rows
//   part 3  dual pass on identity rows (generic leaf prox, no stencil)
// and, for parts 0..2, a second time with -DPB_STENCIL_SLAB=1: the same kernels with the halo
// protocol of the slab decomposition compiled in (SLAB = true).  The single-GPU instantiations
// carry none of it (no extra registers, branches or barriers).
#include <initializer_list>
#include "pb_stencil.cuh"
#include "pb_stencil_staged.cuh"

#include <algorithm>
#include <cstdlib>

#ifndef PB_STENCIL_PART
#error "compile with -DPB_STENCIL_PART=<0..3>"
#endif
#ifndef PB_STENCIL_SLAB
#define PB_STENCIL_SLAB 0
#endif

namespace pb {

constexpr bool kSlab = PB_STENCIL_SLAB != 0;

// Every launch function exists in two flavours with distinct names (plain functions, so that no TU
// can implicitly instantiate the other flavour with its own kernels): <name>_single is compiled in
// the PB_STENCIL_SLAB=0 objects, <name>_slab in the PB_STENCIL_SLAB=1 objects.
#if PB_STENCIL_SLAB
#define PB_FLAVOUR(name) name##_slab
#else
#define PB_FLAVOUR(name) name##_single
#endif

#define PB_DECLARE_PRIMAL(name)                                                                          \
  unsigned name(Context* ctx, const GradGeom& g0, bool three_d, const ProxDesc& d, const float* x,        \
                const float* y, const float* y_prev, ScaleRef T, const PdhgState* st, bool kty_zero,      \
                bool ktyprev_zero, bool check, double* partials, float* x_out, bool dry_run)
#define PB_DECLARE_DUAL(name)                                                                            \
  unsigned name(Context* ctx, const GradGeom& g0, bool three_d, const ProxDesc& d, const float* y,        \
                const float* x_new, const float* x_old, ScaleRef S, const PdhgState* st, bool kxprev_zero, \
                bool check, double* partials, float* y_out, bool dry_run)
PB_DECLARE_PRIMAL(stencil_primal1_launch_single);
PB_DECLARE_PRIMAL(stencil_primal1_launch_slab);
PB_DECLARE_PRIMAL(stencil_primal_simplex_launch_single);
PB_DECLARE_PRIMAL(stencil_primal_simplex_launch_slab);
PB_DECLARE_DUAL(stencil_dual_norm2_launch_single);
PB_DECLARE_DUAL(stencil_dual_norm2_launch_slab);

unsigned stencil_dual_identity_launch(Context* ctx, const GradGeom& g, const ProxDesc& d, const float* y,
                                      const float* x_new, const float* x_old, ScaleRef S, const PdhgState* st,
                                      bool kxprev_zero, bool check, double* partials, float* y_out,
                                      bool dry_run);

static inline GradGeom with_vec(GradGeom g, int vec) {
  g.q = g.ny / vec;
  g.div_q = FastDiv(g.q);
  g.div_nx = FastDiv(g.nx);
  g.div_L = FastDiv(g.L);
  return g;
}

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

static inline unsigned grid_threads(size_t threads) {
  return (unsigned)((threads + kStencilBlock - 1) / kStencilBlock);
}

// per-pixel label groups: operands staged through shared memory (pb_stencil_staged.cuh)
static inline unsigned staged_grid(size_t threads) {
  return (unsigned)((threads + kStagedBlock - 1) / kStagedBlock);
}
template <class Kernel>
static bool staged_configure(Kernel kernel, size_t smem) {
  // dynamic shared memory beyond 48 KB has to be opted into once per kernel
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess;
}

// cooperative 16-byte staging (pb_stencil_staged.cuh): plain iterations, CTAs aligned with image columns
[[maybe_unused]] static bool staged_coop_ok(const GradGeom& g, bool check, std::initializer_list<const void*> arrays) {
  static const bool enabled = [] { const char* e = getenv("PB_STAGED_COOP"); return !e || atoi(e) != 0; }();
  (void)check;
  if (!enabled || g.ny % kStagedBlock != 0 || g.q != g.ny || g.plane % 4 != 0 || g.nxny % 4 != 0 ||
      (g.has_id && g.id_row % 4 != 0))
    return false;
  if ((g.halo.has_left || g.halo.has_right) &&
      ((reinterpret_cast<uintptr_t>(g.halo.in_a) | reinterpret_cast<uintptr_t>(g.halo.in_b)) & 15u))
    return false;
  for (const void* a : arrays)
    if (reinterpret_cast<uintptr_t>(a) & 15u) return false;
  return true;
}

#if PB_STENCIL_PART == 0

#if !PB_STENCIL_SLAB
StencilPlan plan_stencil(const std::vector<std::shared_ptr<Block>>& blocks, size_t nrows, size_t ncols) {
  StencilPlan plan;
  const Block* grad = nullptr;
  const Block* ident = nullptr;
  for (auto& b : blocks) {
    if (b->kind() == kBlockZero) continue;
    if ((b->kind() == kBlockGradient2D || b->kind() == kBlockGradient3D) && !grad) grad = b.get();
    else if (b->kind() == kBlockDiags && !ident) ident = b.get();
    else return plan;
  }
  if (!grad) return plan;
  const BlockDesc gd = grad->desc();
  if (gd.label_first || gd.row != 0 || gd.col != 0 || gd.ncols != ncols) return plan;
  plan.three_d = grad->kind() == kBlockGradient3D;
  GradGeom& g = plan.geom;
  g.nx = gd.nx; g.ny = gd.ny; g.L = gd.L; g.nxny = gd.nx * gd.ny; g.plane = gd.plane;
  if (ident) {
    // exactly  f * I  over all columns, directly below the gradient rows
    const BlockDesc id = ident->desc();
    if (id.ndiags != 1 || id.col != 0 || id.ncols != gd.ncols || id.nrows != gd.ncols ||
        id.row != gd.nrows)
      return plan;
    long long ofs = 0;
    float fac = 0.f;
    if (cudaMemcpy(&ofs, id.offsets, sizeof(ofs), cudaMemcpyDeviceToHost) != cudaSuccess) return plan;
    if (cudaMemcpy(&fac, id.factors, sizeof(fac), cudaMemcpyDeviceToHost) != cudaSuccess) return plan;
    if (ofs != 0) return plan;
    g.has_id = 1;
    g.id_row = id.row;
    g.id_factor = fac;
    if (nrows < (size_t)id.row + id.nrows) return plan;
  }
  plan.ok = true;
  return plan;
}
#endif  // !PB_STENCIL_SLAB

template <int VEC, int KIND, int FN, bool THREE_D, bool HAS_ID>
static void primal1_launch(Context* ctx, unsigned grid, const GradGeom& g, const ProxDesc& d, const float* x,
                           const float* y, const float* y_prev, ScaleRef T, const PdhgState* st,
                           bool kty_zero, bool ktyprev_zero, bool check, double* partials, float* x_out) {
  if (check)
    grad_primal_kernel<VEC, 1, KIND, FN, THREE_D, HAS_ID, true, kSlab><<<grid, kStencilBlock, 0, ctx->stream>>>(
        g, d, x, y, y_prev, T, st, kty_zero, ktyprev_zero, partials, x_out);
  else
    grad_primal_kernel<VEC, 1, KIND, FN, THREE_D, HAS_ID, false, kSlab><<<grid, kStencilBlock, 0, ctx->stream>>>(
        g, d, x, y, y_prev, T, st, kty_zero, ktyprev_zero, partials, x_out);
}

template <int VEC, int KIND, int FN>
static void primal1_geom(Context* ctx, unsigned grid, const GradGeom& g, bool three_d, const ProxDesc& d,
                         const float* x, const float* y, const float* y_prev, ScaleRef T, const PdhgState* st,
                         bool kty_zero, bool ktyprev_zero, bool check, double* partials, float* x_out) {
#define PB_ARGS ctx, grid, g, d, x, y, y_prev, T, st, kty_zero, ktyprev_zero, check, partials, x_out
  if (three_d) {
    if (g.has_id) primal1_launch<VEC, KIND, FN, true, true>(PB_ARGS);
    else primal1_launch<VEC, KIND, FN, true, false>(PB_ARGS);
  } else {
    if (g.has_id) primal1_launch<VEC, KIND, FN, false, true>(PB_ARGS);
    else primal1_launch<VEC, KIND, FN, false, false>(PB_ARGS);
  }
#undef PB_ARGS
}

#if !PB_STENCIL_SLAB
unsigned stencil_primal_launch(Context* ctx, const StencilPlan& plan, const ProxDesc& d, const float* x,
                               const float* y, const float* y_prev, ScaleRef T, const PdhgState* st,
                               bool kty_zero, bool ktyprev_zero, bool check, double* partials, float* x_out,
                               bool dry_run) {
  if (!plan.ok || d.index != 0) return 0;
  const GradGeom& g0 = plan.geom;
  const bool slab = g0.halo.has_left || g0.halo.has_right;
#define PB_ARGS ctx, g0, plan.three_d, d, x, y, y_prev, T, st, kty_zero, ktyprev_zero, check, partials, x_out, dry_run
  if (d.kind == kProxSimplex)
    return slab ? stencil_primal_simplex_launch_slab(PB_ARGS) : stencil_primal_simplex_launch_single(PB_ARGS);
  if (d.kind != kProxElem1D && d.kind != kProxZero) return 0;
  return slab ? stencil_primal1_launch_slab(PB_ARGS) : stencil_primal1_launch_single(PB_ARGS);
#undef PB_ARGS
}
#endif  // !PB_STENCIL_SLAB

PB_DECLARE_PRIMAL(PB_FLAVOUR(stencil_primal1_launch)) {
  if (d.dim != 1 || d.count != g0.plane) return 0;
  bool vec4 = (g0.ny % 4 == 0) && aligned16(x) && aligned16(y) && aligned16(y_prev) && aligned16(x_out) &&
              (!T.ptr || aligned16(T.ptr)) && (!g0.has_id || g0.id_row % 4 == 0);
  for (int k = 0; k < 7; ++k)
    if (d.coeffs.ptr[k] && !aligned16(d.coeffs.ptr[k])) vec4 = false;
  if (g0.halo.has_left && vec4 && !aligned16(g0.halo.out)) vec4 = false;
  const int vec = vec4 ? 4 : 1;
  GradGeom g = with_vec(g0, vec);
  g.halo.n_edge_ctas = count_edge_ctas(g.q, g.L);
  const unsigned grid = grid_threads((size_t)g.q * g.nx * g.L);
  if (dry_run || grid == 0) return grid;
#define PB_ARGS ctx, grid, g, three_d, d, x, y, y_prev, T, st, kty_zero, ktyprev_zero, check, partials, x_out
  // Function1D members with their own instantiation (the data terms of the reference's examples:
  // quadratic for ROF, abs for TV-L1); every other member dispatches at run time (FN = -1)
  if (d.kind == kProxElem1D) {
    if (d.fn == PB_FUN_SQUARE) {
      if (vec == 4) primal1_geom<4, kProxElem1D, PB_FUN_SQUARE>(PB_ARGS); else primal1_geom<1, kProxElem1D, PB_FUN_SQUARE>(PB_ARGS);
    } else if (d.fn == PB_FUN_ABS) {
      if (vec == 4) primal1_geom<4, kProxElem1D, PB_FUN_ABS>(PB_ARGS); else primal1_geom<1, kProxElem1D, PB_FUN_ABS>(PB_ARGS);
    } else {
      if (vec == 4) primal1_geom<4, kProxElem1D, -1>(PB_ARGS); else primal1_geom<1, kProxElem1D, -1>(PB_ARGS);
    }
  } else {
    if (vec == 4) primal1_geom<4, kProxZero, -1>(PB_ARGS); else primal1_geom<1, kProxZero, -1>(PB_ARGS);
  }
#undef PB_ARGS
  PB_CHECK_LAUNCH();
  ctx->launches++;
  return grid;
}

#if !PB_STENCIL_SLAB
unsigned stencil_dual_launch(Context* ctx, const StencilPlan& plan, const ProxDesc& d, const float* y,
                             const float* x_new, const float* x_old, ScaleRef S, const PdhgState* st,
                             bool kxprev_zero, bool check, double* partials, float* y_out, bool dry_run) {
  if (!plan.ok) return 0;
  const GradGeom& g = plan.geom;
  const uint32_t grad_rows = (plan.three_d ? 3u : 2u) * g.plane;
  if (d.index == 0 && d.kind == kProxNorm2 && (size_t)d.count * d.dim == grad_rows) {
    if (g.halo.has_left || g.halo.has_right)
      return stencil_dual_norm2_launch_slab(ctx, g, plan.three_d, d, y, x_new, x_old, S, st, kxprev_zero,
                                            check, partials, y_out, dry_run);
    return stencil_dual_norm2_launch_single(ctx, g, plan.three_d, d, y, x_new, x_old, S, st, kxprev_zero,
                                            check, partials, y_out, dry_run);
  }
  if (g.has_id && d.index == g.id_row && (size_t)d.count * d.dim == g.plane)
    return stencil_dual_identity_launch(ctx, g, d, y, x_new, x_old, S, st, kxprev_zero, check, partials,
                                        y_out, dry_run);
  return 0;
}
#endif  // !PB_STENCIL_SLAB

#elif PB_STENCIL_PART == 1

template <int CAPL, bool HAS_ID>
static void simplex_launch(Context* ctx, unsigned grid, const GradGeom& g, const ProxDesc& d, const float* x,
                           const float* y, const float* y_prev, ScaleRef T, const PdhgState* st,
                           bool kty_zero, bool ktyprev_zero, bool check, double* partials, float* x_out) {
  if (check)
    grad_primal_kernel<1, CAPL, kProxSimplex, -1, false, HAS_ID, true, kSlab><<<grid, kStencilBlock, 0, ctx->stream>>>(
        g, d, x, y, y_prev, T, st, kty_zero, ktyprev_zero, partials, x_out);
  else
    grad_primal_kernel<1, CAPL, kProxSimplex, -1, false, HAS_ID, false, kSlab><<<grid, kStencilBlock, 0, ctx->stream>>>(
        g, d, x, y, y_prev, T, st, kty_zero, ktyprev_zero, partials, x_out);
}

template <int CAPL, bool HAS_ID, bool CHECK>
static bool simplex_staged_launch_k(Context* ctx, unsigned grid, const GradGeom& g, const ProxDesc& d, const float* x,
                                    const float* y, const float* y_prev, float Tval, const PdhgState* st,
                                    bool ktyprev_zero, double* partials, float* x_out) {
  constexpr int LC = CAPL < kStagedChunk ? CAPL : kStagedChunk;
  if constexpr (LC == 4) {
    if (staged_coop_ok(g, CHECK, {x, y, y_prev, x_out})) {
      auto coop = grad_primal_simplex_staged_kernel<CAPL, LC, HAS_ID, CHECK, kSlab, true>;
      const size_t csmem = primal_staged_smem(CAPL, LC, HAS_ID, CHECK, true);
      static const bool cok = staged_configure(coop, csmem);
      if (cok) {
        coop<<<grid, kStagedBlock, csmem, ctx->stream>>>(g, d, x, y, y_prev, Tval, st, ktyprev_zero ? 1 : 0, partials,
                                                         x_out);
        return true;
      }
      cudaGetLastError();
    }
  }
  auto kernel = grad_primal_simplex_staged_kernel<CAPL, LC, HAS_ID, CHECK, kSlab>;
  const size_t smem = primal_staged_smem(CAPL, LC, HAS_ID, CHECK);   // sized for the y_prev operands as well
  static const bool ok = staged_configure(kernel, smem);
  if (!ok) { cudaGetLastError(); return false; }
  kernel<<<grid, kStagedBlock, smem, ctx->stream>>>(g, d, x, y, y_prev, Tval, st, ktyprev_zero ? 1 : 0, partials,
                                                    x_out);
  return true;
}

template <int CAPL>
static bool simplex_staged_launch(Context* ctx, unsigned grid, const GradGeom& g, const ProxDesc& d, const float* x,
                                  const float* y, const float* y_prev, float Tval, const PdhgState* st,
                                  bool ktyprev_zero, bool check, double* partials, float* x_out) {
#define PB_ARGS ctx, grid, g, d, x, y, y_prev, Tval, st, ktyprev_zero, partials, x_out
  if (g.has_id) return check ? simplex_staged_launch_k<CAPL, true, true>(PB_ARGS) : simplex_staged_launch_k<CAPL, true, false>(PB_ARGS);
  return check ? simplex_staged_launch_k<CAPL, false, true>(PB_ARGS) : simplex_staged_launch_k<CAPL, false, false>(PB_ARGS);
#undef PB_ARGS
}

PB_DECLARE_PRIMAL(PB_FLAVOUR(stencil_primal_simplex_launch)) {
  // simplex over the labels of a pixel: planar, count = nx*ny, dim = L (2-D gradient only)
  if (three_d || d.interleaved || d.moreau || d.count != g0.nxny || d.dim != g0.L || g0.L < 2 || g0.L > 32)
    return 0;
  GradGeom g = with_vec(g0, 1);
  const int cap = g.L <= 4 ? 4 : g.L <= 8 ? 8 : g.L <= 16 ? 16 : 32;
  // operands staged through shared memory (every iteration but the first, uniform T)
  if (!kty_zero && !T.ptr) {
    const unsigned sgrid = staged_grid((size_t)g.q * g.nx);
    if (dry_run || sgrid == 0) return sgrid;
    g.halo.n_edge_ctas = staged_grid(g.q);
    bool launched = false;
#define PB_ARGS ctx, sgrid, g, d, x, y, y_prev, T.val, st, ktyprev_zero, check, partials, x_out
    switch (cap) {
      case 4: launched = simplex_staged_launch<4>(PB_ARGS); break;
      case 8: launched = simplex_staged_launch<8>(PB_ARGS); break;
      case 16: launched = simplex_staged_launch<16>(PB_ARGS); break;
      default: launched = simplex_staged_launch<32>(PB_ARGS); break;
    }
#undef PB_ARGS
    if (launched) {
      PB_CHECK_LAUNCH();
      ctx->launches++;
      return sgrid;
    }
  }
  g.halo.n_edge_ctas = count_edge_ctas(g.q, 1);
  const unsigned grid = grid_threads((size_t)g.q * g.nx);
  if (dry_run || grid == 0) return grid;
#define PB_ARGS ctx, grid, g, d, x, y, y_prev, T, st, kty_zero, ktyprev_zero, check, partials, x_out
#define PB_CASE(C) \
  case C: if (g.has_id) simplex_launch<C, true>(PB_ARGS); else simplex_launch<C, false>(PB_ARGS); break;
  switch (cap) { PB_CASE(4) PB_CASE(8) PB_CASE(16) PB_CASE(32) }
#undef PB_CASE
#undef PB_ARGS
  PB_CHECK_LAUNCH();
  ctx->launches++;
  return grid;
}

#elif PB_STENCIL_PART == 2

template <int CAPL, int FN, bool CHECK>
static bool dual_staged_launch_k(Context* ctx, unsigned grid, const GradGeom& g, const ProxDesc& d, const float* y,
                                 const float* x_new, const float* x_old, float Sval, const PdhgState* st,
                                 bool kxprev_zero, double* partials, float* y_out) {
  constexpr int LC = CAPL < kStagedChunk ? CAPL : kStagedChunk;
  if constexpr (LC == 4) {
    if (staged_coop_ok(g, CHECK, {y, x_new, x_old, y_out})) {
      auto coop = grad_dual_norm2_staged_kernel<CAPL, LC, FN, CHECK, kSlab, true>;
      const size_t csmem = dual_staged_smem(CAPL, LC, CHECK, true);
      static const bool cok = staged_configure(coop, csmem);
      if (cok) {
        coop<<<grid, kStagedBlock, csmem, ctx->stream>>>(g, d, y, x_new, x_old, Sval, st, kxprev_zero ? 1 : 0, partials,
                                                         y_out);
        return true;
      }
      cudaGetLastError();
    }
  }
  auto kernel = grad_dual_norm2_staged_kernel<CAPL, LC, FN, CHECK, kSlab>;
  const size_t smem = dual_staged_smem(CAPL, LC, CHECK);
  static const bool ok = staged_configure(kernel, smem);
  if (!ok) { cudaGetLastError(); return false; }
  kernel<<<grid, kStagedBlock, smem, ctx->stream>>>(g, d, y, x_new, x_old, Sval, st, kxprev_zero ? 1 : 0, partials,
                                                    y_out);
  return true;
}

template <int CAPL>
static bool dual_staged_launch(Context* ctx, unsigned grid, const GradGeom& g, const ProxDesc& d, const float* y,
                               const float* x_new, const float* x_old, float Sval, const PdhgState* st,
                               bool kxprev_zero, bool check, double* partials, float* y_out) {
#define PB_ARGS ctx, grid, g, d, y, x_new, x_old, Sval, st, kxprev_zero, partials, y_out
  if (d.fn == PB_FUN_IND_LEQ0)
    return check ? dual_staged_launch_k<CAPL, PB_FUN_IND_LEQ0, true>(PB_ARGS) : dual_staged_launch_k<CAPL, PB_FUN_IND_LEQ0, false>(PB_ARGS);
  return check ? dual_staged_launch_k<CAPL, -1, true>(PB_ARGS) : dual_staged_launch_k<CAPL, -1, false>(PB_ARGS);
#undef PB_ARGS
}

template <int VEC, int CAPL, int FN, bool THREE_D>
static void dual_launch_fn(Context* ctx, unsigned grid, const GradGeom& g, const ProxDesc& d, const float* y,
                           const float* x_new, const float* x_old, ScaleRef S, const PdhgState* st,
                           bool kxprev_zero, bool check, double* partials, float* y_out) {
  if (check)
    grad_dual_norm2_kernel<VEC, CAPL, FN, THREE_D, true, kSlab><<<grid, kStencilBlock, 0, ctx->stream>>>(
        g, d, y, x_new, x_old, S, st, kxprev_zero, partials, y_out);
  else
    grad_dual_norm2_kernel<VEC, CAPL, FN, THREE_D, false, kSlab><<<grid, kStencilBlock, 0, ctx->stream>>>(
        g, d, y, x_new, x_old, S, st, kxprev_zero, partials, y_out);
}

// ind_leq0 (projection onto norm balls, the f* of TV) and abs (TV given as f, through Moreau) get
// their own instantiation; other Function1D members dispatch at run time
template <int VEC, int CAPL, bool THREE_D>
static void dual_launch(Context* ctx, unsigned grid, const GradGeom& g, const ProxDesc& d, const float* y,
                        const float* x_new, const float* x_old, ScaleRef S, const PdhgState* st,
                        bool kxprev_zero, bool check, double* partials, float* y_out) {
  if (d.fn == PB_FUN_IND_LEQ0)
    dual_launch_fn<VEC, CAPL, PB_FUN_IND_LEQ0, THREE_D>(ctx, grid, g, d, y, x_new, x_old, S, st, kxprev_zero, check, partials, y_out);
  else if (d.fn == PB_FUN_ABS)
    dual_launch_fn<VEC, CAPL, PB_FUN_ABS, THREE_D>(ctx, grid, g, d, y, x_new, x_old, S, st, kxprev_zero, check, partials, y_out);
  else
    dual_launch_fn<VEC, CAPL, -1, THREE_D>(ctx, grid, g, d, y, x_new, x_old, S, st, kxprev_zero, check, partials, y_out);
}

PB_DECLARE_DUAL(PB_FLAVOUR(stencil_dual_norm2_launch)) {
  if (d.interleaved) return 0;
  const uint32_t ncomp = three_d ? 3u : 2u;
  const bool per_voxel = d.count == g0.plane && d.dim == ncomp;
  const bool per_pixel = !three_d && g0.L > 1 && d.count == g0.nxny && d.dim == ncomp * g0.L && g0.L <= 32;
  if (!per_voxel && !per_pixel) return 0;
  bool vec4 = (g0.ny % 4 == 0) && aligned16(y) && aligned16(x_new) && aligned16(x_old) && aligned16(y_out) &&
              (!S.ptr || aligned16(S.ptr)) && (g0.plane % 4 == 0);
  for (int k = 0; k < 7; ++k)
    if (d.coeffs.ptr[k] && !aligned16(d.coeffs.ptr[k])) vec4 = false;
  if (per_pixel && g0.L > 4) vec4 = false;             // keep the group within the register budget
  if (g0.halo.has_right && vec4 && !aligned16(g0.halo.out)) vec4 = false;
  // per-pixel groups over more than 4 labels, scalar weights, uniform Sigma on these rows: operands staged
  // through shared memory (pb_stencil_staged.cuh)
  bool scalar_coeffs = !d.moreau && !S.ptr;
  for (int k = 0; k < 7; ++k) scalar_coeffs = scalar_coeffs && !d.coeffs.ptr[k];
  if (per_pixel && g0.L > 4 && scalar_coeffs) {
    GradGeom gs = with_vec(g0, 1);
    const unsigned sgrid = staged_grid((size_t)gs.q * gs.nx);
    if (dry_run || sgrid == 0) return sgrid;
    gs.halo.n_edge_ctas = staged_grid(gs.q);
    bool launched = false;
#define PB_ARGS ctx, sgrid, gs, d, y, x_new, x_old, S.val, st, kxprev_zero, check, partials, y_out
    if (gs.L <= 8) launched = dual_staged_launch<8>(PB_ARGS);
    else if (gs.L <= 16) launched = dual_staged_launch<16>(PB_ARGS);
    else launched = dual_staged_launch<32>(PB_ARGS);
#undef PB_ARGS
    if (launched) {
      PB_CHECK_LAUNCH();
      ctx->launches++;
      return sgrid;
    }
  }
  const int vec = vec4 ? 4 : 1;
  GradGeom g = with_vec(g0, vec);
  g.halo.n_edge_ctas = count_edge_ctas(g.q, per_voxel ? g.L : 1u);
  const unsigned grid = grid_threads((size_t)g.q * g.nx * (per_voxel ? g.L : 1u));
  if (dry_run || grid == 0) return grid;
#define PB_ARGS ctx, grid, g, d, y, x_new, x_old, S, st, kxprev_zero, check, partials, y_out
  if (per_voxel) {
    if (three_d) { if (vec == 4) dual_launch<4, 1, true>(PB_ARGS); else dual_launch<1, 1, true>(PB_ARGS); }
    else { if (vec == 4) dual_launch<4, 1, false>(PB_ARGS); else dual_launch<1, 1, false>(PB_ARGS); }
  } else {
    const int cap = g.L <= 2 ? 2 : g.L <= 4 ? 4 : g.L <= 8 ? 8 : g.L <= 16 ? 16 : 32;
    if (vec == 4) {
      if (cap == 2) dual_launch<4, 2, false>(PB_ARGS); else dual_launch<4, 4, false>(PB_ARGS);
    } else {
      switch (cap) {
        case 2: dual_launch<1, 2, false>(PB_ARGS); break;
        case 4: dual_launch<1, 4, false>(PB_ARGS); break;
        case 8: dual_launch<1, 8, false>(PB_ARGS); break;
        case 16: dual_launch<1, 16, false>(PB_ARGS); break;
        default: dual_launch<1, 32, false>(PB_ARGS); break;
      }
    }
  }
#undef PB_ARGS
  PB_CHECK_LAUNCH();
  ctx->launches++;
  return grid;
}

#elif PB_STENCIL_PART == 3

template <int CAP, int KIND = -1>
static void ident_launch_k(Context* ctx, unsigned grid, const GradGeom& g, const ProxDesc& d, const float* y,
                           const float* x_new, const float* x_old, ScaleRef S, const PdhgState* st,
                           bool kxprev_zero, bool check, double* partials, float* y_out) {
  if (check) {
    IdentityDualSource<CAP, true> src{y, x_new, x_old, S, st, g.id_factor, g.id_row, kxprev_zero, partials};
    prox_pass_kernel<CAP, IdentityDualSource<CAP, true>, KIND><<<grid, kBlock, 0, ctx->stream>>>(d, src, y_out, S, false);
  } else {
    IdentityDualSource<CAP, false> src{y, x_new, x_old, S, st, g.id_factor, g.id_row, kxprev_zero, partials};
    if constexpr (CAP == 2 && KIND == kProxEpiQuad) {
      // (x, y) pairs, planar: four pairs per thread with 128-bit loads / stores when the rows are aligned
      static const bool vec4 = [] { const char* e = getenv("PB_IDENT_VEC4"); return !e || atoi(e) != 0; }();
      auto aligned = [](const float* ptr, size_t off) { return (reinterpret_cast<uintptr_t>(ptr + off) & 15u) == 0; };
      const size_t e0 = d.index, e1 = (size_t)d.index + d.count;
      if (vec4 && d.dim == 2 && !S.ptr && d.count % 4 == 0 && aligned(y, e0) && aligned(y, e1) && aligned(y_out, e0) &&
          aligned(y_out, e1) && aligned(x_new, e0 - g.id_row) && aligned(x_new, e1 - g.id_row) &&
          (kxprev_zero || (aligned(x_old, e0 - g.id_row) && aligned(x_old, e1 - g.id_row)))) {
        const unsigned g4 = (unsigned)std::min<size_t>(grid_for(d.count / 4), (size_t)grid);
        prox_pass_pairs4_kernel<IdentityDualSource<CAP, false>, KIND><<<g4, kBlock, 0, ctx->stream>>>(d, src, y_out, S.val,
                                                                                                      false);
        return;
      }
    }
    prox_pass_kernel<CAP, IdentityDualSource<CAP, false>, KIND><<<grid, kBlock, 0, ctx->stream>>>(d, src, y_out, S, false);
  }
}

template <int CAP>
static void ident_launch(Context* ctx, unsigned grid, const GradGeom& g, const ProxDesc& d, const float* y,
                         const float* x_new, const float* x_old, ScaleRef S, const PdhgState* st,
                         bool kxprev_zero, bool check, double* partials, float* y_out) {
  // the lifted multilabel energy's identity rows carry the epigraph projection on (x, y) pairs: compiled without
  // the run-time prox dispatch (whose dead cases cost registers and local memory, profiles/r01_lifting.md)
  if (CAP == 2 && d.kind == kProxEpiQuad)
    ident_launch_k<CAP, kProxEpiQuad>(ctx, grid, g, d, y, x_new, x_old, S, st, kxprev_zero, check, partials, y_out);
  else
    ident_launch_k<CAP, -1>(ctx, grid, g, d, y, x_new, x_old, S, st, kxprev_zero, check, partials, y_out);
}

unsigned stencil_dual_identity_launch(Context* ctx, const GradGeom& g, const ProxDesc& d, const float* y,
                                      const float* x_new, const float* x_old, ScaleRef S, const PdhgState* st,
                                      bool kxprev_zero, bool check, double* partials, float* y_out,
                                      bool dry_run) {
  const int cap = dim_cap(d.dim, d.kind);
  if (cap == 0 || cap > 8) return 0;
  const unsigned grid = (unsigned)std::min<size_t>(grid_for(d.count), (size_t)ctx->num_sms * 16);
  if (dry_run || d.count == 0) return d.count ? grid : 0;
#define PB_ARGS ctx, grid, g, d, y, x_new, x_old, S, st, kxprev_zero, check, partials, y_out
  switch (cap) {
    case 1: ident_launch<1>(PB_ARGS); break;
    case 2: ident_launch<2>(PB_ARGS); break;
    case 4: ident_launch<4>(PB_ARGS); break;
    default: ident_launch<8>(PB_ARGS); break;
  }
#undef PB_ARGS
  PB_CHECK_LAUNCH();
  ctx->launches++;
  return grid;
}

#endif

}  // namespace pb
