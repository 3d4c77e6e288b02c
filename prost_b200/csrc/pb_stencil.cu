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

// Each launches the pass of a prox that stencil_primal_cover / stencil_dual_cover assigned to it and returns the
// grid; the caller (stencil_primal_launch / stencil_dual_launch) checks and counts the launch.
unsigned stencil_primal1_launch_single(Context*, const GradGeom&, bool three_d, const ProxDesc&, const PrimalPass&);
unsigned stencil_primal1_launch_slab(Context*, const GradGeom&, bool three_d, const ProxDesc&, const PrimalPass&);
unsigned stencil_primal_simplex_launch_single(Context*, const GradGeom&, bool three_d, const ProxDesc&,
                                              const PrimalPass&);
unsigned stencil_primal_simplex_launch_slab(Context*, const GradGeom&, bool three_d, const ProxDesc&,
                                            const PrimalPass&);
unsigned stencil_dual_norm2_launch_single(Context*, const GradGeom&, bool three_d, const ProxDesc&, const DualPass&);
unsigned stencil_dual_norm2_launch_slab(Context*, const GradGeom&, bool three_d, const ProxDesc&, const DualPass&);
unsigned stencil_dual_identity_launch(Context*, const GradGeom&, const ProxDesc&, const DualPass&);

// the plan's geometry for threads of `vec` rows, with the pass's halo
static inline GradGeom with_vec(GradGeom g, int vec, const SlabHalo* halo) {
  if (halo) g.halo = *halo;
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
// threads of `vec` rows over n_l label planes of every column
static inline unsigned stencil_grid(const GradGeom& g, int vec, uint32_t n_l) {
  return grid_threads((size_t)(g.ny / vec) * g.nx * n_l);
}

// per-pixel label groups: operands staged through shared memory (pb_stencil_staged.cuh)
static inline unsigned staged_grid(size_t threads) {
  return (unsigned)((threads + kStagedBlock - 1) / kStagedBlock);
}

static inline unsigned identity_grid(const Context* ctx, const ProxDesc& d) {
  return (unsigned)std::min<size_t>(grid_for(d.count), (size_t)ctx->num_sms * 16);
}
template <class Kernel>
static bool staged_configure(Kernel kernel, size_t smem) {
  // dynamic shared memory beyond 48 KB has to be opted into once per kernel
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess;
}

// cooperative 16-byte staging (pb_stencil_staged.cuh): plain iterations, CTAs aligned with image columns
[[maybe_unused]] static bool staged_coop_ok(const GradGeom& g, std::initializer_list<const void*> arrays) {
  static const bool enabled = [] { const char* e = getenv("PB_STAGED_COOP"); return !e || atoi(e) != 0; }();
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

// the launch site of grad_primal_kernel (parts 0 and 1)
template <int VEC, int CAPL, int KIND, int FN, bool THREE_D, bool HAS_ID>
static void primal_launch(Context* ctx, unsigned grid, const GradGeom& g, const ProxDesc& d, const PrimalPass& p) {
  auto kernel = p.check ? grad_primal_kernel<VEC, CAPL, KIND, FN, THREE_D, HAS_ID, true, kSlab>
                        : grad_primal_kernel<VEC, CAPL, KIND, FN, THREE_D, HAS_ID, false, kSlab>;
  check_partials_fit(p.check, grid, p.partials_cap);
  kernel<<<grid, kStencilBlock, 0, ctx->stream>>>(g, d, p.x, p.y, p.y_prev, p.T, p.st, p.kty_zero, p.ktyprev_zero,
                                                  p.partials, p.x_out);
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

template <int VEC, int KIND, int FN>
static void primal1_geom(Context* ctx, unsigned grid, const GradGeom& g, bool three_d, const ProxDesc& d,
                         const PrimalPass& p) {
  if (three_d) {
    if (g.has_id) primal_launch<VEC, 1, KIND, FN, true, true>(ctx, grid, g, d, p);
    else primal_launch<VEC, 1, KIND, FN, true, false>(ctx, grid, g, d, p);
  } else {
    if (g.has_id) primal_launch<VEC, 1, KIND, FN, false, true>(ctx, grid, g, d, p);
    else primal_launch<VEC, 1, KIND, FN, false, false>(ctx, grid, g, d, p);
  }
}

#if !PB_STENCIL_SLAB
unsigned stencil_primal_cover(const StencilPlan& plan, const ProxDesc& d) {
  const GradGeom& g = plan.geom;
  if (!plan.ok || d.index != 0 || d.count == 0) return 0;
  // one-element groups over every voxel
  if (d.kind == kProxElem1D || d.kind == kProxZero) return d.dim == 1 && d.count == g.plane ? stencil_grid(g, 1, g.L) : 0;
  // simplex over the labels of a pixel: planar, count = nx*ny, dim = L (2-D gradient only)
  if (d.kind == kProxSimplex && !plan.three_d && !d.interleaved && !d.moreau && d.count == g.nxny && d.dim == g.L &&
      g.L >= 2 && g.L <= 32)
    return std::max(staged_grid(g.nxny), stencil_grid(g, 1, 1));
  return 0;
}

unsigned stencil_dual_cover(const Context* ctx, const StencilPlan& plan, const ProxDesc& d) {
  const GradGeom& g = plan.geom;
  if (!plan.ok || d.count == 0) return 0;
  const uint32_t ncomp = plan.three_d ? 3u : 2u;
  if (d.index == 0 && d.kind == kProxNorm2 && (size_t)d.count * d.dim == ncomp * g.plane) {
    if (d.interleaved) return 0;
    // the gradient components of a voxel
    if (d.count == g.plane && d.dim == ncomp) return stencil_grid(g, 1, g.L);
    // those of all labels of a pixel (2-D); staged through shared memory above 4 labels
    if (plan.three_d || g.L <= 1 || g.L > 32 || d.count != g.nxny || d.dim != ncomp * g.L) return 0;
    return g.L > 4 ? std::max(staged_grid(g.nxny), stencil_grid(g, 1, 1)) : stencil_grid(g, 1, 1);
  }
  // the identity rows: a leaf prox held in at most 8 registers
  const int cap = dim_cap(d.dim, d.kind);
  if (g.has_id && d.index == g.id_row && (size_t)d.count * d.dim == g.plane && cap > 0 && cap <= 8)
    return identity_grid(ctx, d);
  return 0;
}

unsigned stencil_primal_launch(Context* ctx, const StencilPlan& plan, const ProxDesc& d, const PrimalPass& p) {
  if (!stencil_primal_cover(plan, d)) return 0;
  // slab kernels where the pass has a neighbour; a communicator of one rank runs the single-GPU ones
  const bool slab = p.halo && (p.halo->has_left || p.halo->has_right);
  const unsigned grid =
      d.kind == kProxSimplex
          ? (slab ? stencil_primal_simplex_launch_slab : stencil_primal_simplex_launch_single)(ctx, plan.geom,
                                                                                               plan.three_d, d, p)
          : (slab ? stencil_primal1_launch_slab : stencil_primal1_launch_single)(ctx, plan.geom, plan.three_d, d, p);
  PB_CHECK_LAUNCH();
  ctx->launches++;
  return grid;
}
#endif  // !PB_STENCIL_SLAB

unsigned PB_FLAVOUR(stencil_primal1_launch)(Context* ctx, const GradGeom& g0, bool three_d, const ProxDesc& d,
                                            const PrimalPass& p) {
  bool vec4 = (g0.ny % 4 == 0) && aligned16(p.x) && aligned16(p.y) && aligned16(p.y_prev) && aligned16(p.x_out) &&
              (!p.T.ptr || aligned16(p.T.ptr)) && (!g0.has_id || g0.id_row % 4 == 0);
  for (int k = 0; k < 7; ++k)
    if (d.coeffs.ptr[k] && !aligned16(d.coeffs.ptr[k])) vec4 = false;
  if (p.halo && p.halo->has_left && vec4 && !aligned16(p.halo->out)) vec4 = false;
  const int vec = vec4 ? 4 : 1;
  GradGeom g = with_vec(g0, vec, p.halo);
  g.halo.n_edge_ctas = count_edge_ctas(g.q, g.L);
  const unsigned grid = stencil_grid(g, vec, g.L);
  // Function1D members with their own instantiation (the data terms of the reference's examples:
  // quadratic for ROF, abs for TV-L1); every other member dispatches at run time (FN = -1)
  if (d.kind == kProxElem1D) {
    if (d.fn == PB_FUN_SQUARE) {
      if (vec == 4) primal1_geom<4, kProxElem1D, PB_FUN_SQUARE>(ctx, grid, g, three_d, d, p);
      else primal1_geom<1, kProxElem1D, PB_FUN_SQUARE>(ctx, grid, g, three_d, d, p);
    } else if (d.fn == PB_FUN_ABS) {
      if (vec == 4) primal1_geom<4, kProxElem1D, PB_FUN_ABS>(ctx, grid, g, three_d, d, p);
      else primal1_geom<1, kProxElem1D, PB_FUN_ABS>(ctx, grid, g, three_d, d, p);
    } else {
      if (vec == 4) primal1_geom<4, kProxElem1D, -1>(ctx, grid, g, three_d, d, p);
      else primal1_geom<1, kProxElem1D, -1>(ctx, grid, g, three_d, d, p);
    }
  } else {
    if (vec == 4) primal1_geom<4, kProxZero, -1>(ctx, grid, g, three_d, d, p);
    else primal1_geom<1, kProxZero, -1>(ctx, grid, g, three_d, d, p);
  }
  return grid;
}

#if !PB_STENCIL_SLAB
unsigned stencil_dual_launch(Context* ctx, const StencilPlan& plan, const ProxDesc& d, const DualPass& p) {
  if (!stencil_dual_cover(ctx, plan, d)) return 0;
  const bool slab = p.halo && (p.halo->has_left || p.halo->has_right);
  // Norm2 on the gradient rows, otherwise the identity rows
  const unsigned grid =
      d.index == 0 && d.kind == kProxNorm2
          ? (slab ? stencil_dual_norm2_launch_slab : stencil_dual_norm2_launch_single)(ctx, plan.geom, plan.three_d, d, p)
          : stencil_dual_identity_launch(ctx, plan.geom, d, p);
  PB_CHECK_LAUNCH();
  ctx->launches++;
  return grid;
}
#endif  // !PB_STENCIL_SLAB

#elif PB_STENCIL_PART == 1

template <int CAPL, bool HAS_ID, bool CHECK>
static bool simplex_staged_launch_k(Context* ctx, unsigned grid, const GradGeom& g, const ProxDesc& d,
                                    const PrimalPass& p) {
  constexpr int LC = CAPL < kStagedChunk ? CAPL : kStagedChunk;
  auto launch = [&](auto kernel, size_t smem) {
    check_partials_fit(CHECK, grid, p.partials_cap);
    kernel<<<grid, kStagedBlock, smem, ctx->stream>>>(g, d, p.x, p.y, p.y_prev, p.T.val, p.st, p.ktyprev_zero ? 1 : 0,
                                                      p.partials, p.x_out);
  };
  if constexpr (LC == 4) {
    if (staged_coop_ok(g, {p.x, p.y, p.y_prev, p.x_out})) {
      auto coop = grad_primal_simplex_staged_kernel<CAPL, LC, HAS_ID, CHECK, kSlab, true>;
      const size_t csmem = primal_staged_smem(CAPL, LC, HAS_ID, CHECK, true);
      static const bool cok = staged_configure(coop, csmem);
      if (cok) {
        launch(coop, csmem);
        return true;
      }
      cudaGetLastError();
    }
  }
  auto kernel = grad_primal_simplex_staged_kernel<CAPL, LC, HAS_ID, CHECK, kSlab>;
  const size_t smem = primal_staged_smem(CAPL, LC, HAS_ID, CHECK);   // sized for the y_prev operands as well
  static const bool ok = staged_configure(kernel, smem);
  if (!ok) { cudaGetLastError(); return false; }
  launch(kernel, smem);
  return true;
}

template <int CAPL>
static bool simplex_staged_launch(Context* ctx, unsigned grid, const GradGeom& g, const ProxDesc& d,
                                  const PrimalPass& p) {
  if (g.has_id)
    return p.check ? simplex_staged_launch_k<CAPL, true, true>(ctx, grid, g, d, p)
                   : simplex_staged_launch_k<CAPL, true, false>(ctx, grid, g, d, p);
  return p.check ? simplex_staged_launch_k<CAPL, false, true>(ctx, grid, g, d, p)
                 : simplex_staged_launch_k<CAPL, false, false>(ctx, grid, g, d, p);
}

unsigned PB_FLAVOUR(stencil_primal_simplex_launch)(Context* ctx, const GradGeom& g0, bool, const ProxDesc& d,
                                                   const PrimalPass& p) {
  GradGeom g = with_vec(g0, 1, p.halo);
  const int cap = g.L <= 4 ? 4 : g.L <= 8 ? 8 : g.L <= 16 ? 16 : 32;
  // operands staged through shared memory (every iteration but the first, uniform T)
  if (!p.kty_zero && !p.T.ptr) {
    const unsigned sgrid = staged_grid(g.nxny);
    g.halo.n_edge_ctas = staged_grid(g.q);
    bool launched = false;
    switch (cap) {
      case 4: launched = simplex_staged_launch<4>(ctx, sgrid, g, d, p); break;
      case 8: launched = simplex_staged_launch<8>(ctx, sgrid, g, d, p); break;
      case 16: launched = simplex_staged_launch<16>(ctx, sgrid, g, d, p); break;
      default: launched = simplex_staged_launch<32>(ctx, sgrid, g, d, p); break;
    }
    if (launched) return sgrid;
  }
  g.halo.n_edge_ctas = count_edge_ctas(g.q, 1);
  const unsigned grid = stencil_grid(g, 1, 1);
#define PB_CASE(C)                                                                      \
  case C:                                                                               \
    if (g.has_id) primal_launch<1, C, kProxSimplex, -1, false, true>(ctx, grid, g, d, p); \
    else primal_launch<1, C, kProxSimplex, -1, false, false>(ctx, grid, g, d, p);         \
    break;
  switch (cap) { PB_CASE(4) PB_CASE(8) PB_CASE(16) PB_CASE(32) }
#undef PB_CASE
  return grid;
}

#elif PB_STENCIL_PART == 2

template <int CAPL, int FN, bool CHECK>
static bool dual_staged_launch_k(Context* ctx, unsigned grid, const GradGeom& g, const ProxDesc& d,
                                 const DualPass& p) {
  constexpr int LC = CAPL < kStagedChunk ? CAPL : kStagedChunk;
  auto launch = [&](auto kernel, size_t smem) {
    check_partials_fit(CHECK, grid, p.partials_cap);
    kernel<<<grid, kStagedBlock, smem, ctx->stream>>>(g, d, p.y, p.x_new, p.x_old, p.S.val, p.st, p.kxprev_zero ? 1 : 0,
                                                      p.partials, p.y_out);
  };
  if constexpr (LC == 4) {
    if (staged_coop_ok(g, {p.y, p.x_new, p.x_old, p.y_out})) {
      auto coop = grad_dual_norm2_staged_kernel<CAPL, LC, FN, CHECK, kSlab, true>;
      const size_t csmem = dual_staged_smem(CAPL, LC, CHECK, true);
      static const bool cok = staged_configure(coop, csmem);
      if (cok) {
        launch(coop, csmem);
        return true;
      }
      cudaGetLastError();
    }
  }
  auto kernel = grad_dual_norm2_staged_kernel<CAPL, LC, FN, CHECK, kSlab>;
  const size_t smem = dual_staged_smem(CAPL, LC, CHECK);
  static const bool ok = staged_configure(kernel, smem);
  if (!ok) { cudaGetLastError(); return false; }
  launch(kernel, smem);
  return true;
}

template <int CAPL>
static bool dual_staged_launch(Context* ctx, unsigned grid, const GradGeom& g, const ProxDesc& d, const DualPass& p) {
  if (d.fn == PB_FUN_IND_LEQ0)
    return p.check ? dual_staged_launch_k<CAPL, PB_FUN_IND_LEQ0, true>(ctx, grid, g, d, p)
                   : dual_staged_launch_k<CAPL, PB_FUN_IND_LEQ0, false>(ctx, grid, g, d, p);
  return p.check ? dual_staged_launch_k<CAPL, -1, true>(ctx, grid, g, d, p)
                 : dual_staged_launch_k<CAPL, -1, false>(ctx, grid, g, d, p);
}

// the launch site of grad_dual_norm2_kernel
template <int VEC, int CAPL, int FN, bool THREE_D>
static void dual_launch_fn(Context* ctx, unsigned grid, const GradGeom& g, const ProxDesc& d, const DualPass& p) {
  auto kernel = p.check ? grad_dual_norm2_kernel<VEC, CAPL, FN, THREE_D, true, kSlab>
                        : grad_dual_norm2_kernel<VEC, CAPL, FN, THREE_D, false, kSlab>;
  check_partials_fit(p.check, grid, p.partials_cap);
  kernel<<<grid, kStencilBlock, 0, ctx->stream>>>(g, d, p.y, p.x_new, p.x_old, p.S, p.st, p.kxprev_zero, p.partials,
                                                  p.y_out);
}

// ind_leq0 (projection onto norm balls, the f* of TV) and abs (TV given as f, through Moreau) get
// their own instantiation; other Function1D members dispatch at run time
template <int VEC, int CAPL, bool THREE_D>
static void dual_launch(Context* ctx, unsigned grid, const GradGeom& g, const ProxDesc& d, const DualPass& p) {
  if (d.fn == PB_FUN_IND_LEQ0) dual_launch_fn<VEC, CAPL, PB_FUN_IND_LEQ0, THREE_D>(ctx, grid, g, d, p);
  else if (d.fn == PB_FUN_ABS) dual_launch_fn<VEC, CAPL, PB_FUN_ABS, THREE_D>(ctx, grid, g, d, p);
  else dual_launch_fn<VEC, CAPL, -1, THREE_D>(ctx, grid, g, d, p);
}

unsigned PB_FLAVOUR(stencil_dual_norm2_launch)(Context* ctx, const GradGeom& g0, bool three_d, const ProxDesc& d,
                                               const DualPass& p) {
  const bool per_voxel = d.count == g0.plane && d.dim == (three_d ? 3u : 2u), per_pixel = !per_voxel;
  bool vec4 = (g0.ny % 4 == 0) && aligned16(p.y) && aligned16(p.x_new) && aligned16(p.x_old) && aligned16(p.y_out) &&
              (!p.S.ptr || aligned16(p.S.ptr)) && (g0.plane % 4 == 0);
  for (int k = 0; k < 7; ++k)
    if (d.coeffs.ptr[k] && !aligned16(d.coeffs.ptr[k])) vec4 = false;
  if (per_pixel && g0.L > 4) vec4 = false;             // keep the group within the register budget
  if (p.halo && p.halo->has_right && vec4 && !aligned16(p.halo->out)) vec4 = false;
  // per-pixel groups over more than 4 labels, scalar weights, uniform Sigma on these rows: operands staged
  // through shared memory (pb_stencil_staged.cuh)
  bool scalar_coeffs = !d.moreau && !p.S.ptr;
  for (int k = 0; k < 7; ++k) scalar_coeffs = scalar_coeffs && !d.coeffs.ptr[k];
  if (per_pixel && g0.L > 4 && scalar_coeffs) {
    GradGeom gs = with_vec(g0, 1, p.halo);
    const unsigned sgrid = staged_grid(gs.nxny);
    gs.halo.n_edge_ctas = staged_grid(gs.q);
    bool launched = false;
    if (gs.L <= 8) launched = dual_staged_launch<8>(ctx, sgrid, gs, d, p);
    else if (gs.L <= 16) launched = dual_staged_launch<16>(ctx, sgrid, gs, d, p);
    else launched = dual_staged_launch<32>(ctx, sgrid, gs, d, p);
    if (launched) return sgrid;
  }
  const int vec = vec4 ? 4 : 1;
  GradGeom g = with_vec(g0, vec, p.halo);
  g.halo.n_edge_ctas = count_edge_ctas(g.q, per_voxel ? g.L : 1u);
  const unsigned grid = stencil_grid(g, vec, per_voxel ? g.L : 1u);
  if (per_voxel) {
    if (three_d) {
      if (vec == 4) dual_launch<4, 1, true>(ctx, grid, g, d, p);
      else dual_launch<1, 1, true>(ctx, grid, g, d, p);
    } else {
      if (vec == 4) dual_launch<4, 1, false>(ctx, grid, g, d, p);
      else dual_launch<1, 1, false>(ctx, grid, g, d, p);
    }
  } else {
    const int cap = g.L <= 2 ? 2 : g.L <= 4 ? 4 : g.L <= 8 ? 8 : g.L <= 16 ? 16 : 32;
    if (vec == 4) {
      if (cap == 2) dual_launch<4, 2, false>(ctx, grid, g, d, p);
      else dual_launch<4, 4, false>(ctx, grid, g, d, p);
    } else {
      switch (cap) {
        case 2: dual_launch<1, 2, false>(ctx, grid, g, d, p); break;
        case 4: dual_launch<1, 4, false>(ctx, grid, g, d, p); break;
        case 8: dual_launch<1, 8, false>(ctx, grid, g, d, p); break;
        case 16: dual_launch<1, 16, false>(ctx, grid, g, d, p); break;
        default: dual_launch<1, 32, false>(ctx, grid, g, d, p); break;
      }
    }
  }
  return grid;
}

#elif PB_STENCIL_PART == 3

template <int CAP, int KIND = -1>
static void ident_launch_k(Context* ctx, unsigned grid, const GradGeom& g, const ProxDesc& d, const DualPass& p) {
  if (p.check) {
    IdentityDualSource<CAP, true> src{p.y, p.x_new, p.x_old, p.S, p.st, g.id_factor, g.id_row, p.kxprev_zero, p.partials};
    prox_pass_kernel<CAP, IdentityDualSource<CAP, true>, KIND><<<grid, kBlock, 0, ctx->stream>>>(d, src, p.y_out, p.S,
                                                                                                  false);
  } else {
    IdentityDualSource<CAP, false> src{p.y, p.x_new, p.x_old, p.S, p.st, g.id_factor, g.id_row, p.kxprev_zero, p.partials};
    if constexpr (CAP == 2 && KIND == kProxEpiQuad) {
      // (x, y) pairs, planar: four pairs per thread with 128-bit loads / stores when the rows are aligned
      static const bool vec4 = [] { const char* e = getenv("PB_IDENT_VEC4"); return !e || atoi(e) != 0; }();
      auto aligned = [](const float* ptr, size_t off) { return (reinterpret_cast<uintptr_t>(ptr + off) & 15u) == 0; };
      const size_t e0 = d.index, e1 = (size_t)d.index + d.count;
      if (vec4 && d.dim == 2 && !p.S.ptr && d.count % 4 == 0 && aligned(p.y, e0) && aligned(p.y, e1) &&
          aligned(p.y_out, e0) && aligned(p.y_out, e1) && aligned(p.x_new, e0 - g.id_row) &&
          aligned(p.x_new, e1 - g.id_row) &&
          (p.kxprev_zero || (aligned(p.x_old, e0 - g.id_row) && aligned(p.x_old, e1 - g.id_row)))) {
        const unsigned g4 = (unsigned)std::min<size_t>(grid_for(d.count / 4), (size_t)grid);
        prox_pass_pairs4_kernel<IdentityDualSource<CAP, false>, KIND><<<g4, kBlock, 0, ctx->stream>>>(d, src, p.y_out,
                                                                                                      p.S.val, false);
        return;
      }
    }
    prox_pass_kernel<CAP, IdentityDualSource<CAP, false>, KIND><<<grid, kBlock, 0, ctx->stream>>>(d, src, p.y_out, p.S,
                                                                                                   false);
  }
}

template <int CAP>
static void ident_launch(Context* ctx, unsigned grid, const GradGeom& g, const ProxDesc& d, const DualPass& p) {
  // the lifted multilabel energy's identity rows carry the epigraph projection on (x, y) pairs: compiled without
  // the run-time prox dispatch (whose dead cases cost registers and local memory, profiles/r01_lifting.md)
  if (CAP == 2 && d.kind == kProxEpiQuad) ident_launch_k<CAP, kProxEpiQuad>(ctx, grid, g, d, p);
  else ident_launch_k<CAP, -1>(ctx, grid, g, d, p);
}

unsigned stencil_dual_identity_launch(Context* ctx, const GradGeom& g, const ProxDesc& d, const DualPass& p) {
  const unsigned grid = identity_grid(ctx, d);
  check_partials_fit(p.check, grid, p.partials_cap);
  switch (dim_cap(d.dim, d.kind)) {
    case 1: ident_launch<1>(ctx, grid, g, d, p); break;
    case 2: ident_launch<2>(ctx, grid, g, d, p); break;
    case 4: ident_launch<4>(ctx, grid, g, d, p); break;
    default: ident_launch<8>(ctx, grid, g, d, p); break;
  }
  return grid;
}

#endif

}  // namespace pb
