// pb_fused_cap.cu -- one translation unit per register capacity PB_CAP (1,2,4,...,64) so the
// fused-pass instantiations compile in parallel.  See pb_fused.cuh for the kernels.
#include "pb_fused.cuh"

#ifndef PB_CAP
#error "compile with -DPB_CAP=<1|2|4|8|16|32|64>"
#endif

namespace pb {

template <int CAP, bool CHECK>
static void primal_launch(Context* ctx, unsigned grid, const ProxDesc& d, const BlockList& bl, const PrimalPass& p) {
  PrimalSource<CAP, CHECK> src;
  src.x = p.x; src.y = p.y; src.y_prev = p.y_prev; src.T = p.T; src.st = p.st; src.bl = bl;
  src.kty_zero = p.kty_zero; src.ktyprev_zero = p.ktyprev_zero; src.partials = p.partials;
  prox_pass_kernel<CAP, PrimalSource<CAP, CHECK>><<<grid, kBlock, 0, ctx->stream>>>(d, src, p.x_out, p.T, false);
}

template <int CAP, bool CHECK>
static void dual_launch(Context* ctx, unsigned grid, const ProxDesc& d, const BlockList& bl, const DualPass& p) {
  DualSource<CAP, CHECK> src;
  src.y = p.y; src.x_new = p.x_new; src.x_old = p.x_old; src.S = p.S; src.st = p.st; src.bl = bl;
  src.kxprev_zero = p.kxprev_zero; src.partials = p.partials;
  prox_pass_kernel<CAP, DualSource<CAP, CHECK>><<<grid, kBlock, 0, ctx->stream>>>(d, src, p.y_out, p.S, false);
}

template <int CAP>
void fused_primal_cap(Context* ctx, unsigned grid, const ProxDesc& d, const BlockList& bl, const PrimalPass& p) {
  if (p.check) primal_launch<CAP, true>(ctx, grid, d, bl, p);
  else primal_launch<CAP, false>(ctx, grid, d, bl, p);
}

template <int CAP>
void fused_dual_cap(Context* ctx, unsigned grid, const ProxDesc& d, const BlockList& bl, const DualPass& p) {
  if (p.check) dual_launch<CAP, true>(ctx, grid, d, bl, p);
  else dual_launch<CAP, false>(ctx, grid, d, bl, p);
}

template void fused_primal_cap<PB_CAP>(Context*, unsigned, const ProxDesc&, const BlockList&, const PrimalPass&);
template void fused_dual_cap<PB_CAP>(Context*, unsigned, const ProxDesc&, const BlockList&, const DualPass&);

}  // namespace pb
