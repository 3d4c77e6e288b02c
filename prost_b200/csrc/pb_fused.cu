// pb_fused.cu -- dispatch of the generic fused PDHG passes (pb_fused.cuh) to the per-capacity
// translation units (pb_fused_cap.cu).
#include "pb_fused.cuh"

#include <algorithm>

namespace pb {

// defined in pb_fused_cap.cu and instantiated there for one CAP per translation unit
template <int CAP> void fused_primal_cap(Context*, unsigned grid, const ProxDesc&, const BlockList&, const PrimalPass&);
template <int CAP> void fused_dual_cap(Context*, unsigned grid, const ProxDesc&, const BlockList&, const DualPass&);

unsigned fused_grid(Context* ctx, const ProxDesc& d) {
  // grid-stride: enough CTAs for 8 resident per SM, never more than the work
  return (unsigned)std::min<size_t>(grid_for(d.count), (size_t)ctx->num_sms * 8);
}

unsigned fused_primal_launch(Context* ctx, const ProxDesc& d, const BlockList& bl, const PrimalPass& p) {
  if (d.count == 0) return 0;
  const unsigned grid = fused_grid(ctx, d);
  check_partials_fit(p.check, grid, p.partials_cap);
#define PB_CASE(N) case N: fused_primal_cap<N>(ctx, grid, d, bl, p); break;
  switch (dim_cap(d.dim, d.kind)) {
    PB_CASE(1) PB_CASE(2) PB_CASE(4) PB_CASE(8) PB_CASE(16) PB_CASE(32) PB_CASE(64)
    default: fail(PB_ERR_UNSUPPORTED, "fused pass: group dimension too large");
  }
#undef PB_CASE
  PB_CHECK_LAUNCH();
  ctx->launches++;
  return grid;
}

unsigned fused_dual_launch(Context* ctx, const ProxDesc& d, const BlockList& bl, const DualPass& p) {
  if (d.count == 0) return 0;
  const unsigned grid = fused_grid(ctx, d);
  check_partials_fit(p.check, grid, p.partials_cap);
#define PB_CASE(N) case N: fused_dual_cap<N>(ctx, grid, d, bl, p); break;
  switch (dim_cap(d.dim, d.kind)) {
    PB_CASE(1) PB_CASE(2) PB_CASE(4) PB_CASE(8) PB_CASE(16) PB_CASE(32) PB_CASE(64)
    default: fail(PB_ERR_UNSUPPORTED, "fused pass: group dimension too large");
  }
#undef PB_CASE
  PB_CHECK_LAUNCH();
  ctx->launches++;
  return grid;
}

}  // namespace pb
