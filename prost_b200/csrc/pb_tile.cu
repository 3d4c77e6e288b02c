// pb_tile.cu -- one whole PDHG iteration in ONE pass over HBM for planar 2-D gradient operators.
//
// The two-pass schedule (pb_stencil.cuh) moves 44 B per pixel and iteration for ROF: the dual pass
// re-reads x+, x and y that the primal pass had in registers a moment earlier.  Here an owned tile of
// TX x TY pixels is computed in two phases:
//   phase A  x+ = prox_g(x - tau T K^T y) on the tile PLUS one halo column (x = cx+TX) and one
//            halo row vector (y = cy+TY): the forward differences of the dual step need x+ there.  x+ and
//            x of the extended tile go to shared memory; the tile's own x+ is written to HBM.  A tile at the
//            image bottom has no tile below it and owns its halo row vector as well.
//   phase B  y+ = prox_f*(y + sigma S ((1+theta) K x+ - theta K x)) on the tile, with K x+ and K x
//            taken from shared memory.
// HBM traffic per pixel: read y (2), x, f; write x+, y+ (2) = 7 floats = 28 B instead of 44 B; the
// halo re-computation costs (TX+1)(TY+4)/(TX TY) - 1 = 6.6 % extra arithmetic (TX = 31, TY = 124) and loads
// that hit L2 (they are a neighbouring tile's primary loads).  The halo values of x+ are recomputed with
// exactly the same instructions as in the tile that owns them, so the result is bit-identical to the
// two-pass kernels, which in turn follow the reference operation by operation
// (backend_pdhg.cu:38-70, 311-381; block_gradient2d.cu:25-139).
//
// Used on iterations that neither refresh the residuals nor need the iteration-0 special cases
// (K^T y := 0, K x_prev := 0); those run the two-pass kernels on the same ping-pong buffers.
#include "pb_stencil.cuh"

#include <cuda.h>

#include <algorithm>
#include <cstdlib>
#include <map>
#include <mutex>
#include <tuple>

namespace pb {

namespace {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, void* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// ---- tensor maps (host) ------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    cudaGetLastError();
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}

// 3-D map over a planar float array [planes][nx][ny] (ny contiguous) with a (rows x cols x 1) box
bool tensor_map_for(const float* base, uint32_t ny, uint32_t nx, uint32_t planes, uint32_t box_rows,
                    uint32_t box_cols, CUtensorMap& out) {
  typedef std::tuple<const void*, uint32_t, uint32_t, uint32_t, uint32_t, uint32_t> Key;
  static std::map<Key, CUtensorMap> cache;
  static std::mutex mu;
  const Key key(base, ny, nx, planes, box_rows, box_cols);
  std::lock_guard<std::mutex> lock(mu);
  auto it = cache.find(key);
  if (it != cache.end()) { out = it->second; return true; }
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return false;
  const cuuint64_t dims[3] = {ny, nx, planes};
  const cuuint64_t strides[2] = {(cuuint64_t)ny * 4, (cuuint64_t)ny * nx * 4};
  const cuuint32_t box[3] = {box_rows, box_cols, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  CUtensorMap m;
  const CUresult r = enc(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return false;
  if (cache.size() > 256) cache.clear();
  cache[key] = m;
  out = m;
  return true;
}

// ---- persistent TMA ring ------------------------------------------------------------------------------
// A kernel that loads one tile, computes it and exits alternates between waiting for memory and computing:
// with plain loads or one-shot TMA boxes such kernels reached 72 % / 68 % of HBM bandwidth, against 84 %
// for this one (profiles/r01_tile.md).  Here ONE CTA of 1024 threads stays resident per SM and walks over
// tiles; the operand boxes of the next two tiles are always in flight (two shared-memory stages filled by
// TMA, completion signalled on mbarriers), so HBM streams continuously while the 32 warps compute the
// current tile.
//   computed x+ region 32 columns x 128 rows = 1024 row vectors = exactly one per thread;
//   owned tile         31 columns x 124 rows (the last column / 4 rows are the halo of the neighbours);
//                      the bottom tile of a tile column owns all 128 rows: nothing below it needs them, and
//                      the forward difference of the image's last row is 0 anyway, so at ny = 4096 the
//                      33 tile rows cover 32 x 124 + 128 rows exactly instead of leaving a 34th with 4 rows.
// Walk: CTA b takes tiles b, b + grid, b + 2 grid, ... (label plane, then tile column, then tile row).  Plain
// single-GPU launches alternate between this order and its reverse, so that the first tiles a launch reads are
// the last ones the previous launch wrote, while those are still in L2.
// Operand boxes per tile at owned-tile origin (cy, cx); out-of-image elements are zero-filled by TMA,
// which is exactly the K^T boundary rule for x = -1 and y = -1:
//   p1    (cy,   cx-1)   33 columns x 128 rows   gx component of y incl. the left neighbour column
//   p2    (cy-4, cx)     32 columns x 132 rows   gy component of y incl. row cy-1 (16-byte aligned)
//   x, f  (cy,   cx)     32 columns x 128 rows   primal iterate and data term
// There is no CTA-wide barrier in the loop: warp w computes column w; its dual step only needs the
// x+ of columns w and w+1, so it waits on column w+1's mbarrier; a stage is recycled when all 32
// warps have arrived on its `empty` barrier, which warp 31 (it owns the halo column and has no dual
// work) observes before it issues the next TMA loads.
constexpr int kRingThreads = 1024;
constexpr int kRingCols = 32, kRingRows = 128;          // computed region
constexpr int kRingTX = kRingCols - 1, kRingTY = kRingRows - 4;   // owned tile
constexpr int kRingR2 = kRingRows + 4;                  // p2 box rows (starts 4 rows early)
constexpr int kRingP1Bytes = (kRingCols + 1) * kRingRows * 4;
constexpr int kRingP2Bytes = kRingCols * kRingR2 * 4;
constexpr int kRingXBytes = kRingCols * kRingRows * 4;
// stage contents: [p1][p2][x][f]; residual-refresh launches (CHECK) stage the previous dual iterate's
// boxes [q1][q2] instead of f (which they read from global memory) so that two stages still fit
constexpr int kRingStageBytes = 2 * (kRingP1Bytes + kRingP2Bytes) + kRingXBytes;
constexpr int kRingStages = 2;
constexpr int kRingOffXn = kRingStages * kRingStageBytes;            // x+ tiles, one per stage
constexpr int kRingOffBar = kRingOffXn + kRingStages * kRingXBytes;
// mbarriers: full[stage] (TMA bytes landed), empty[stage] (all 32 warps done with the stage),
// col_ready[stage][column] (that column's x+ is in shared memory).  Every barrier belongs to one stage, so
// it can never run more than one phase ahead of a waiter (a stage is only refilled after ALL warps left it).
constexpr int kRingSmemBytes = kRingOffBar + (2 * kRingStages + kRingStages * kRingCols) * 8 + 64;
static_assert(kRingP1Bytes % 128 == 0 && kRingP2Bytes % 128 == 0 && kRingXBytes % 128 == 0, "TMA alignment");

__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  // try_wait suspends the warp in hardware until the phase completes or the time hint (ns) expires,
  // so a waiting warp costs (almost) no issue slots; the loop only covers the time-out case
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n selp.u32 %0, 1, 0, p;\n}"
        : "=r"(done) : "r"(smem_u32(bar)), "r"(parity), "r"(1000000u) : "memory");
  }
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- flag-in-data halo lines (RingHalo, pb_comm.cuh) -----------------------------------------------------------
// four rows = two 16-byte lines {v0, seq, v1, seq} {v2, seq, v3, seq}; volatile accesses go to L2, the point of
// coherence for the neighbour's NVLink stores
__device__ __forceinline__ void ll_ld_line(const uint4* p, uint4& v) {
  asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
}
// the four rows of sequence number `seq`: spins until all four tags match (gives up after ~2 s, no GPU hang)
__device__ __forceinline__ void ll_wait_load4(const uint4* p, unsigned seq, float (&o)[4], int* error) {
  uint4 a, b;
  unsigned long long t0 = 0;
  for (unsigned spins = 0;; ++spins) {
    ll_ld_line(p, a);
    ll_ld_line(p + 1, b);
    if (a.y == seq && a.w == seq && b.y == seq && b.w == seq) break;
    if ((spins & 255u) == 255u) {
      if (error && *reinterpret_cast<volatile int*>(error)) break;      // sticky: one timeout poisons the solve
      unsigned long long now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      else if (now - t0 > 2000000000ull) { if (error) atomicExch(error, 1); break; }
    }
  }
  o[0] = __uint_as_float(a.x); o[1] = __uint_as_float(a.z); o[2] = __uint_as_float(b.x); o[3] = __uint_as_float(b.z);
}
// same, with the first poll already issued (lines a, b were loaded before the caller waited for something else)
__device__ __forceinline__ void ll_finish_load4(const uint4* p, unsigned seq, uint4 a, uint4 b, float (&o)[4],
                                                int* error) {
  if (!(a.y == seq && a.w == seq && b.y == seq && b.w == seq)) {
    ll_wait_load4(p, seq, o, error);
    return;
  }
  o[0] = __uint_as_float(a.x); o[1] = __uint_as_float(a.z); o[2] = __uint_as_float(b.x); o[3] = __uint_as_float(b.z);
}
// slot selection without indexing the kernel-parameter arrays dynamically (that would copy them to local memory)
template <class P>
__device__ __forceinline__ P sel3(P const (&a)[3], unsigned k) { return k == 0u ? a[0] : (k == 1u ? a[1] : a[2]); }
template <class P>
__device__ __forceinline__ P sel2(P const (&a)[2], unsigned k) { return k == 0u ? a[0] : a[1]; }
// rows that are known to be there (the slot of an earlier sequence number)
__device__ __forceinline__ void ll_read4(const uint4* p, float (&o)[4]) {
  uint4 a, b;
  ll_ld_line(p, a);
  ll_ld_line(p + 1, b);
  o[0] = __uint_as_float(a.x); o[1] = __uint_as_float(a.z); o[2] = __uint_as_float(b.x); o[3] = __uint_as_float(b.z);
}
__device__ __forceinline__ void ll_store4(uint4* p, const float (&v)[4], unsigned seq) {
  asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(__float_as_uint(v[0])), "r"(seq),
               "r"(__float_as_uint(v[1])), "r"(seq) : "memory");
  asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p + 1), "r"(__float_as_uint(v[2])), "r"(seq),
               "r"(__float_as_uint(v[3])), "r"(seq) : "memory");
}

// PB_RING_TRACE: per launch {first CTA start, last CTA end, longest left-edge halo wait, longest right-edge halo
// wait} in globaltimer ns (atomicMin / atomicMax) at buf[4 * slot]; slot = launch number modulo the buffer length
struct RingTraceSlot {
  unsigned long long* buf = nullptr;   // null: tracing off
  unsigned slot = 0;
};

// CHECK: this iteration refreshes the residuals (backend_pdhg.cu:73-120, 383-436): the same pass also
// gathers K^T y_prev from the previous dual iterate (map_q1 / map_q2) and accumulates the four residual
// sums in double, one (a, b) pair per CTA for each of the two residuals.
// SLAB: the image is a block of columns of a wider one (has_left / has_right neighbours, RingHalo).
template <int FN_G, int FN_F, bool CHECK, bool SLAB>
__global__ void __launch_bounds__(kRingThreads, 1) grad2d_iteration_ring_kernel(
    const __grid_constant__ CUtensorMap map_p1, const __grid_constant__ CUtensorMap map_p2,
    const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_f,
    const __grid_constant__ CUtensorMap map_q1, const __grid_constant__ CUtensorMap map_q2, const GradGeom g,
    const ProxDesc pg, const ProxDesc pf, const float Tval, const float Sval,
    const PdhgState* __restrict__ st, const FastDiv div_per_plane, const FastDiv div_tiles_y,
    const uint32_t n_tiles, const bool reverse, const int ktyprev_zero, double* __restrict__ part_d,
    double* __restrict__ part_p, float* __restrict__ x_out, float* __restrict__ y_out, const uint32_t tiles_x,
    const RingHalo h, const RingTraceSlot trace, const RingFinish fin) {
  extern __shared__ __align__(128) unsigned char smem[];
  // tile -> (label plane, tile column, tile row).  On a slab the left-edge tile column is walked first (its new x
  // column leaves at the start of the launch) and the right-edge one at the first position of the SECOND wave:
  // its tiles need the right neighbour's x column of this very iteration, which that rank's first wave produces.
  // Slabs therefore never walk in reverse.  The producer and the consumers decode the same way.
  const uint32_t right_pos = min(tiles_x - 1u, (gridDim.x + div_tiles_y.d - 1u) / div_tiles_y.d);
  auto decode = [&](uint32_t tile, uint32_t& l, uint32_t& tx, uint32_t& ty) {
    if (!SLAB && reverse) tile = n_tiles - 1u - tile;
    uint32_t rem;
    div_per_plane.divmod(tile, l, rem);
    div_tiles_y.divmod(rem, tx, ty);
    if (SLAB) tx = tx < right_pos ? tx : (tx == right_pos ? tiles_x - 1 : tx - 1);
  };
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + kRingOffBar);
  uint64_t* empty = full + kRingStages;
  uint64_t* col_ready = empty + kRingStages;

  const bool f_vec = pg.coeffs.ptr[1] != nullptr;
  const bool q_boxes = CHECK && !ktyprev_zero;
  const uint32_t stage_tx = kRingP1Bytes + kRingP2Bytes + kRingXBytes +
                            (CHECK ? (q_boxes ? kRingP1Bytes + kRingP2Bytes : 0) : (f_vec ? kRingXBytes : 0));

  auto issue = [&](uint32_t tile, int s) {           // producer lane only
    uint32_t l, tx, ty;
    decode(tile, l, tx, ty);
    const int cx = tx * kRingTX, cy = ty * kRingTY;
    unsigned char* base = smem + s * kRingStageBytes;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&full[s])), "r"(stage_tx)
                 : "memory");
    tma_load_3d(base, &map_p1, &full[s], cy, cx - 1, (int)l);
    tma_load_3d(base + kRingP1Bytes, &map_p2, &full[s], cy - 4, cx, (int)(g.L + l));
    tma_load_3d(base + kRingP1Bytes + kRingP2Bytes, &map_x, &full[s], cy, cx, (int)l);
    if (CHECK) {
      if (q_boxes) {
        tma_load_3d(base + kRingP1Bytes + kRingP2Bytes + kRingXBytes, &map_q1, &full[s], cy, cx - 1, (int)l);
        tma_load_3d(base + 2 * kRingP1Bytes + kRingP2Bytes + kRingXBytes, &map_q2, &full[s], cy - 4, cx,
                    (int)(g.L + l));
      }
    } else if (f_vec) {
      tma_load_3d(base + kRingP1Bytes + kRingP2Bytes + kRingXBytes, &map_f, &full[s], cy, cx, (int)l);
    }
  };

  const bool producer = threadIdx.x == kRingThreads - 32;     // lane 0 of warp 31
  if (producer) {
#pragma unroll
    for (int s = 0; s < kRingStages; ++s) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&full[s])));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 32;" ::"r"(smem_u32(&empty[s])));
    }
    for (int c = 0; c < kRingStages * kRingCols; ++c)
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&col_ready[c])));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    // tensor maps into the descriptor cache while the previous launch drains
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_p1)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_p2)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_x)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_f)) : "memory");
  }
  // Programmatic dependent launch: iteration k+1 is launched while iteration k still runs (its CTAs become
  // resident as SMs free up), so launch latency and this prologue overlap the previous launch's tail; from here
  // on every thread may touch what that launch wrote (iterates, step-size state), hence the wait.  The next
  // launch may be scheduled right away: it blocks at the same point until THIS grid has completed and flushed.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (trace.buf && threadIdx.x == 0) {
    unsigned long long now;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
    atomicMin(trace.buf + 4 * trace.slot, now);
  }
  __syncthreads();
  if (producer) {
#pragma unroll
    for (int s = 0; s < kRingStages; ++s) {
      const uint32_t t = blockIdx.x + s * gridDim.x;
      if (t < n_tiles) issue(t, s);
    }
  }

  const float tau = st->tau, sigma = st->sigma, theta = st->theta;
  Coeffs7 cg, cf;
#pragma unroll
  for (int k = 0; k < 7; ++k) { cg.v[k] = pg.coeffs.val[k]; cf.v[k] = pf.coeffs.val[k]; }
  const bool g_simple = coeffs_simple(cg) && cg.v[2] != 0.f;
  const int fn_g = FN_G >= 0 ? FN_G : pg.fn;
  const float tau_g = effective_tau(tau, Tval, false);
  const int fn_f = FN_F >= 0 ? FN_F : pf.fn;
  const float tau_f = effective_tau(sigma, Sval, false);
  const bool f_simple = coeffs_simple(cf);

  const int col = threadIdx.x >> 5;          // warp = column of the computed region
  const int r0 = (threadIdx.x & 31) * 4;     // lane = row vector
  double acc_d0 = 0.0, acc_d1 = 0.0, acc_p0 = 0.0, acc_p1 = 0.0;
  // residual sums (CHECK): T, Sigma, tau, sigma are uniform here, so the divisions of backend_pdhg.cu:85-88,
  // 109-113 become multiplications by two reciprocals computed once (1 ulp per term, far inside the 1e-4 bar
  // on the residuals); the squares of a thread's four pixels are summed in float before they enter the double
  // accumulators (one conversion per sum instead of one per pixel)
  const float sq_T = sqrtf(Tval), sq_S = sqrtf(Sval);
  const float inv_tau_sq = 1.f / (tau * sq_T), inv_sigma_sq = 1.f / (sigma * sq_S);

  for (uint32_t tile = blockIdx.x, k = 0; tile < n_tiles; tile += gridDim.x, ++k) {
    const int s = k % kRingStages;
    const uint32_t parity = (k / kRingStages) & 1u;
    uint32_t l, tx, ty;
    decode(tile, l, tx, ty);
    const int cx = tx * kRingTX, cy = ty * kRingTY;
    unsigned char* base = smem + s * kRingStageBytes;
    float (*s_p1)[kRingRows] = reinterpret_cast<float (*)[kRingRows]>(base);
    float (*s_p2)[kRingR2] = reinterpret_cast<float (*)[kRingR2]>(base + kRingP1Bytes);
    float (*s_x)[kRingRows] = reinterpret_cast<float (*)[kRingRows]>(base + kRingP1Bytes + kRingP2Bytes);
    float (*s_f)[kRingRows] = reinterpret_cast<float (*)[kRingRows]>(base + kRingP1Bytes + kRingP2Bytes + kRingXBytes);
    float (*s_q1)[kRingRows] = reinterpret_cast<float (*)[kRingRows]>(base + kRingP1Bytes + kRingP2Bytes + kRingXBytes);
    float (*s_q2)[kRingR2] = reinterpret_cast<float (*)[kRingR2]>(base + 2 * kRingP1Bytes + kRingP2Bytes + kRingXBytes);
    float (*s_xn)[kRingRows] = reinterpret_cast<float (*)[kRingRows]>(smem + kRingOffXn + s * kRingXBytes);

    const uint32_t gx = cx + col, gy = cy + r0;
    // this thread's rows belong to the tile (x+ store, dual step, both residual sums); see the owned tile above
    const bool own_rows = r0 < kRingTY || cy + kRingRows >= g.ny;
    const uint32_t plane_off = l * g.nxny;
    // slab edges (warp-uniform): column 0 takes y.gx of column -1 from the left neighbour's halo; the
    // owner of column nx-1 takes x+ / x of column nx from the right neighbour's halo
    const bool left_edge = SLAB && h.has_left && gx == 0;
    const bool right_edge = SLAB && h.has_right && gx == g.nx - 1 && col < kRingTX;
    const uint32_t halo_ll = (((gy < g.ny ? gy : 0u) + l * g.ny) >> 2) * 2u;      // two 16-byte lines per 4 rows
    // first poll of this warp's halo lines before the wait for the operand boxes: a volatile load of lines the
    // neighbour wrote over NVLink takes 1-2 us, which the TMA wait hides
    uint4 pre_a = make_uint4(0u, 0u, 0u, 0u), pre_b = make_uint4(0u, 0u, 0u, 0u);
    const uint4* pre_p = nullptr;
    if (SLAB) {
      if (left_edge && h.y_wait_seq) pre_p = sel3(h.yl_ll, h.y_wait_seq % 3u) + halo_ll;
      else if (right_edge) pre_p = sel2(h.xr_ll, h.x_wait_seq & 1u) + halo_ll;
      if (pre_p) { ll_ld_line(pre_p, pre_a); ll_ld_line(pre_p + 1, pre_b); }
    }
    mbar_wait(&full[s], parity);
    // ---- phase A: x+ at (col, r0..r0+3) of the computed region ------------------------------------------
    if (gx < g.nx) {
      float xo[4], divx[4], o[4], a[4], xn[4];
      // boundary rules as selects on always-valid shared-memory reads (no divergent regions):
      // out-of-image box elements are TMA zero fill == the rule for x = -1 / y = -1 (x - 0 == x exactly)
      VecIO<4>::ld(&s_x[col][r0], xo);
      VecIO<4>::ld(&s_p1[col + 1][r0], divx);
      VecIO<4>::ld(&s_p1[col][r0], a);
      float qa_halo[4] = {0.f, 0.f, 0.f, 0.f};
      if (left_edge) {
        // y.gx of column -1: the left neighbour's previous iteration, row group by row group
        unsigned long long tw0 = 0;
        if (trace.buf) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tw0));
        if (h.y_wait_seq) ll_finish_load4(pre_p, h.y_wait_seq, pre_a, pre_b, a, h.error);
        if (trace.buf) {
          unsigned long long tw1;
          asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tw1));
          atomicMax(trace.buf + 4 * trace.slot + 2, tw1 - tw0);
        }
        // (refresh) the column before it, read BEFORE this thread's x store lets the neighbour move on
        if (CHECK && q_boxes && h.y_wait_seq > 1u) ll_read4(sel3(h.yl_ll, (h.y_wait_seq - 1u) % 3u) + halo_ll, qa_halo);
      }
      VecIO<4>::ld(&s_p2[col][4 + r0], o);
      const float up = s_p2[col][4 + r0 - 1];
      const bool last_col = gx == g.nx - 1 && !(SLAB && h.has_right);
      float divy[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        divx[j] = (last_col ? 0.f : divx[j]) - a[j];
        divy[j] = (gy + j == g.ny - 1) ? 0.f : o[j];
      }
      divy[0] -= up;
#pragma unroll
      for (int j = 1; j < 4; ++j) divy[j] -= o[j - 1];
#pragma unroll
      for (int j = 0; j < 4; ++j) xn[j] = primal_prox_arg(xo[j], tau, Tval, -(divx[j] + divy[j]));
      float bv[4];
      if (f_vec) {
        if (CHECK) {
          // rows beyond the image are never used; clamp the address instead of predicating the load
          const uint32_t gyc = gy < g.ny ? gy : 0u;
          VecIO<4>::ld(pg.coeffs.ptr[1] + gyc + gx * g.ny + plane_off, bv);
        } else {
          VecIO<4>::ld(&s_f[col][r0], bv);
        }
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) bv[j] = cg.v[1];
      }
      if (g_simple) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          xn[j] = scaled_fun_prox_simple(fn_g, xn[j], tau_g, bv[j], cg.v[2], cg.v[5], cg.v[6]);
      } else {
        Coeffs7 c = cg;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          c.v[1] = bv[j];
          xn[j] = elem1d_apply(fn_g, xn[j], tau, Tval, false, c);
        }
      }
      VecIO<4>::st(&s_xn[col][r0], xn);
      if (col < kRingTX && own_rows && gy < g.ny) {
        VecIO<4>::st(x_out + gy + gx * g.ny + plane_off, xn);
        if (left_edge) ll_store4(sel2(h.x_out_ll, h.x_signal_seq & 1u) + halo_ll, xn, h.x_signal_seq);   // -> left neighbour
        if (CHECK) {
          // dual residual on the owned pixels: w^ = (x - x+)/(tau sqrt T) - sqrt T K^T y_prev,
          // diff = w^ + sqrt T K^T y
          float kp[4];
          if (q_boxes) {
            float qx[4], qa[4], qo[4];
            VecIO<4>::ld(&s_q1[col + 1][r0], qx);
            VecIO<4>::ld(&s_q1[col][r0], qa);
            if (left_edge) {
#pragma unroll
              for (int j = 0; j < 4; ++j) qa[j] = qa_halo[j];
            }
            VecIO<4>::ld(&s_q2[col][4 + r0], qo);
            const float qup = s_q2[col][4 + r0 - 1];
            float qy[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              qx[j] = (last_col ? 0.f : qx[j]) - qa[j];
              qy[j] = (gy + j == g.ny - 1) ? 0.f : qo[j];
            }
            qy[0] -= qup;
#pragma unroll
            for (int j = 1; j < 4; ++j) qy[j] -= qo[j - 1];
#pragma unroll
            for (int j = 0; j < 4; ++j) kp[j] = -(qx[j] + qy[j]);
          } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) kp[j] = 0.f;
          }
          float s0 = 0.f, s1 = 0.f;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float kk = -(divx[j] + divy[j]);
            const float w_hat = (xo[j] - xn[j]) * inv_tau_sq - sq_T * kp[j];
            const float diff = w_hat + sq_T * kk;
            s0 += diff * diff;
            s1 += w_hat * w_hat;
          }
          acc_d0 += static_cast<double>(s0);
          acc_d1 += static_cast<double>(s1);
        }
      }
    }
    // publish this column's x+ (one arrival per warp), then wait for the right neighbour's
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(&col_ready[s * kRingCols + col]);
    if (col < kRingTX) mbar_wait(&col_ready[s * kRingCols + col + 1], parity);

    // ---- phase B: y+ at the owned point (col, r0..r0+3) ---------------------------------------------------
    if (col < kRingTX && own_rows && gx < g.nx && gy < g.ny) {
      const uint32_t idx = gy + gx * g.ny + plane_off;
      float arg[2][4];
      float cn[4], co[4], rn[4], ro[4];
      VecIO<4>::ld(&s_xn[col][r0], cn);
      VecIO<4>::ld(&s_x[col][r0], co);
      if (right_edge) {
        // x+ / x of column nx: the right neighbour's column 0 of THIS iteration and of the previous one
        unsigned long long tw0 = 0;
        if (trace.buf) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tw0));
        ll_finish_load4(pre_p, h.x_wait_seq, pre_a, pre_b, rn, h.error);
        if (trace.buf) {
          unsigned long long tw1;
          asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tw1));
          atomicMax(trace.buf + 4 * trace.slot + 3, tw1 - tw0);
        }
        ll_read4(sel2(h.xr_ll, (h.x_wait_seq - 1u) & 1u) + halo_ll, ro);
      } else {
        VecIO<4>::ld(&s_xn[col + 1][r0], rn);
        VecIO<4>::ld(&s_x[col + 1][r0], ro);
      }
      // the row vector below; at r0 = 124 (bottom tile) that is row 0 of column col + 1 <= 31, inside the tile,
      // and last_row discards it
      const float dn = (&s_xn[col][r0])[4], dold = (&s_x[col][r0])[4];
      const bool last_col = gx == g.nx - 1 && !(SLAB && h.has_right), last_row = gy + 4 >= g.ny;
      float k1x[4], k0x[4], k1y[4], k0y[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {          // grad_fwd: 0 on the last column
        k1x[j] = last_col ? 0.f : rn[j] - cn[j];
        k0x[j] = last_col ? 0.f : ro[j] - co[j];
      }
#pragma unroll
      for (int j = 0; j < 3; ++j) { k1y[j] = cn[j + 1] - cn[j]; k0y[j] = co[j + 1] - co[j]; }
      k1y[3] = last_row ? 0.f : dn - cn[3];   // 0 on the last row
      k0y[3] = last_row ? 0.f : dold - co[3];
      float y1[4], y2[4];
      VecIO<4>::ld(&s_p1[col + 1][r0], y1);
      VecIO<4>::ld(&s_p2[col][4 + r0], y2);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        arg[0][j] = dual_prox_arg(y1[j], sigma, Sval, dual_extrapolate(theta, k1x[j], k0x[j]));
        arg[1][j] = dual_prox_arg(y2[j], sigma, Sval, dual_extrapolate(theta, k1y[j], k0y[j]));
      }
      if (f_simple) norm2_lanes<4, 2, true>(fn_f, arg, cf, tau_f);
      else norm2_lanes<4, 2, false>(fn_f, arg, cf, tau_f);
      VecIO<4>::st(y_out + idx, arg[0]);
      VecIO<4>::st(y_out + (size_t)g.L * g.nxny + idx, arg[1]);
      if (right_edge) ll_store4(sel3(h.y_out_ll, h.y_signal_seq % 3u) + halo_ll, arg[0], h.y_signal_seq);   // -> right neighbour
      if (CHECK) {
        // primal residual: z^ = (y - y+)/(sigma sqrt S) + sqrt S ((1+theta) K x+ - theta K x),
        // diff = z^ - sqrt S K x+
        float s0 = 0.f, s1 = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float ex = dual_extrapolate(theta, k1x[j], k0x[j]);
          const float zx = (y1[j] - arg[0][j]) * inv_sigma_sq + sq_S * ex;
          const float dx = zx - sq_S * k1x[j];
          const float ey = dual_extrapolate(theta, k1y[j], k0y[j]);
          const float zy = (y2[j] - arg[1][j]) * inv_sigma_sq + sq_S * ey;
          const float dy = zy - sq_S * k1y[j];
          s0 += dx * dx + dy * dy;
          s1 += zx * zx + zy * zy;
        }
        acc_p0 += static_cast<double>(s0);
        acc_p1 += static_cast<double>(s1);
      }
    }
    // this warp is done with stage s (operand boxes and x+ tile)
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(&empty[s]);
    if (col == kRingCols - 1) {       // warp 31 refills the stage once every warp has left it
      const uint32_t next = tile + kRingStages * gridDim.x;
      if (next < n_tiles) {
        mbar_wait(&empty[s], parity);
        if (producer) issue(next, s);
      }
    }
  }
  if (trace.buf && threadIdx.x == 0) {
    unsigned long long now;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
    atomicMax(trace.buf + 4 * trace.slot + 1, now);
  }
  if (CHECK) {
    block_sum2(acc_d0, acc_d1);
    block_sum2(acc_p0, acc_p1);
    __shared__ unsigned s_last;
    if (threadIdx.x == 0) {
      part_d[2 * blockIdx.x] = acc_d0; part_d[2 * blockIdx.x + 1] = acc_d1;
      part_p[2 * blockIdx.x] = acc_p0; part_p[2 * blockIdx.x + 1] = acc_p1;
      unsigned last = 0;
      if (fin.ticket) {
        __threadfence();
        last = atomicAdd(fin.ticket, 1u) + 1u == gridDim.x ? 1u : 0u;
      }
      s_last = last;
    }
    __syncthreads();
    if (s_last) {
      // last CTA of the launch: every partial pair is visible (ticket + fences); fold in index order
      __threadfence();
      double pa = 0.0, pb = 0.0, da = 0.0, db = 0.0;
      for (unsigned i = threadIdx.x; i < gridDim.x; i += blockDim.x) {
        pa += __ldcg(part_p + 2 * i); pb += __ldcg(part_p + 2 * i + 1);
        da += __ldcg(part_d + 2 * i); db += __ldcg(part_d + 2 * i + 1);
      }
      block_sum2(pa, pb);
      block_sum2(da, db);
      if (threadIdx.x == 0) {
        double sums[4] = {pa, pb, da, db};
        cross_rank_sum4(fin.cross, sums);
        PdhgState ns = *fin.state;
        ns.iteration = fin.iteration;
        pdhg_update(ns, fin.prm, sums, true);
        *fin.state = ns;
        *fin.ticket = 0u;
      }
    }
  }
}

// ---- PB_RING_TRACE=1: launch timeline for scaling experiments (pb_ring_trace_read in the C ABI) ----------------
constexpr unsigned kRingTraceSlots = 4096;
struct RingTrace {
  unsigned long long* buf = nullptr;
  unsigned next = 0;
};
RingTrace& ring_trace() {
  static RingTrace t;
  return t;
}
RingTraceSlot ring_trace_next() {
  RingTraceSlot m;
  static const bool on = [] { const char* e = getenv("PB_RING_TRACE"); return e && atoi(e) != 0; }();
  if (!on) return m;
  RingTrace& t = ring_trace();
  if (!t.buf) {
    if (cudaMalloc(&t.buf, kRingTraceSlots * 4 * sizeof(unsigned long long)) != cudaSuccess) { cudaGetLastError(); return m; }
    std::vector<unsigned long long> init(kRingTraceSlots * 4, 0ull);
    for (unsigned i = 0; i < kRingTraceSlots; ++i) init[4 * i] = ~0ull;
    cudaMemcpy(t.buf, init.data(), init.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice);
  }
  m.buf = t.buf;
  m.slot = t.next++ % kRingTraceSlots;
  return m;
}

// the TMA descriptors of a launch (see the kernel's parameters)
struct RingMaps {
  CUtensorMap mp1, mp2, mx, mf, mq1, mq2;
};

// the ring kernel's tiles: tiles_x * tiles_y owned tiles per label plane, walked by at most one CTA per SM; the
// bottom tile row owns kRingRows rows, the others kRingTY: tiles_y = max(1, ceil((ny - 4) / kRingTY))
struct RingTiles {
  uint32_t x, y;
  uint64_t n;
  explicit RingTiles(const GradGeom& g)
      : x((g.nx + kRingTX - 1) / kRingTX),
        y(g.ny == 0 ? 0 : (std::max(g.ny, (uint32_t)kRingRows) - (kRingRows - kRingTY) + kRingTY - 1) / kRingTY),
        n((uint64_t)x * y * g.L) {}
  unsigned grid(const Context* ctx) const { return (unsigned)std::min<uint64_t>(n, (uint64_t)ctx->num_sms); }
};

// (every instantiation has the same parameters)
template <int FN_G, int FN_F>
auto ring_kernel_fn(bool check, bool slab) {
  return slab ? (check ? grad2d_iteration_ring_kernel<FN_G, FN_F, true, true>
                       : grad2d_iteration_ring_kernel<FN_G, FN_F, false, true>)
              : (check ? grad2d_iteration_ring_kernel<FN_G, FN_F, true, false>
                       : grad2d_iteration_ring_kernel<FN_G, FN_F, false, false>);
}

auto ring_kernel(const ProxDesc& pg, const ProxDesc& pf, bool check, bool slab) {
  const bool leq0 = pf.fn == PB_FUN_IND_LEQ0;
  auto pick = pg.fn == PB_FUN_SQUARE ? (leq0 ? ring_kernel_fn<PB_FUN_SQUARE, PB_FUN_IND_LEQ0> : ring_kernel_fn<PB_FUN_SQUARE, -1>)
            : pg.fn == PB_FUN_ABS    ? (leq0 ? ring_kernel_fn<PB_FUN_ABS, PB_FUN_IND_LEQ0> : ring_kernel_fn<PB_FUN_ABS, -1>)
                                     : (leq0 ? ring_kernel_fn<-1, PB_FUN_IND_LEQ0> : ring_kernel_fn<-1, -1>);
  return pick(check, slab);
}

// returns the number of CTAs (= residual partial pairs per residual when check), 0 if not launched
unsigned ring_launch(Context* ctx, const GradGeom& g, const ProxDesc& pg, const ProxDesc& pf, const TilePass& p) {
  RingMaps m;
  if (!tensor_map_for(p.y, g.ny, g.nx, 2 * g.L, kRingRows, kRingCols + 1, m.mp1)) return 0;
  if (!tensor_map_for(p.y, g.ny, g.nx, 2 * g.L, kRingR2, kRingCols, m.mp2)) return 0;
  if (!tensor_map_for(p.x, g.ny, g.nx, g.L, kRingRows, kRingCols, m.mx)) return 0;
  const float* f = pg.coeffs.ptr[1] ? pg.coeffs.ptr[1] : p.x;    // unused when b is a scalar
  if (!tensor_map_for(f, g.ny, g.nx, g.L, kRingRows, kRingCols, m.mf)) return 0;
  const float* q = (p.check && !p.ktyprev_zero) ? p.y_prev : p.y;  // unused otherwise
  if (!tensor_map_for(q, g.ny, g.nx, 2 * g.L, kRingRows, kRingCols + 1, m.mq1)) return 0;
  if (!tensor_map_for(q, g.ny, g.nx, 2 * g.L, kRingR2, kRingCols, m.mq2)) return 0;
  const RingTiles t(g);
  const unsigned grid = t.grid(ctx);
  check_partials_fit(p.check, grid, p.part_cap);
  RingHalo h;
  if (p.halo) h = *p.halo;
  // programmatic stream serialization: see griddepcontrol in the kernel.  Measured (profiles/r02_scaling.md): the
  // launch-to-launch gap drops from 3.8 to 1.8 us on one GPU, but on slabs the end-of-kernel flush of the
  // NVLink halo stores dominates the gap and early-resident CTAs cost more than they hide (period 54.3 vs
  // 52.9 us at 2 x 2048 columns), so slabs keep plain stream order.
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kRingThreads);
  cfg.dynamicSmemBytes = kRingSmemBytes;
  cfg.stream = ctx->stream;
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr.val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = &attr;
  cfg.numAttrs = p.halo ? 0 : 1;
  const cudaError_t e = cudaLaunchKernelEx(
      &cfg, ring_kernel(pg, pf, p.check, p.halo != nullptr), m.mp1, m.mp2, m.mx, m.mf, m.mq1, m.mq2, g, pg, pf,
      p.T.val, p.S.val, p.st, FastDiv((uint64_t)t.x * t.y), FastDiv(t.y), (uint32_t)t.n, p.reverse, p.ktyprev_zero ? 1 : 0,
      p.part_d, p.part_p, p.x_out, p.y_out, t.x, h, ring_trace_next(), (p.check && p.finish) ? *p.finish : RingFinish());
  if (e != cudaSuccess) { cudaGetLastError(); return 0; }
  return grid;
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace

// copies the trace (up to n launches x 4 values) to the host; returns the number of launches recorded so far
unsigned tile_ring_trace_read(unsigned long long* h_out, unsigned n) {
  RingTrace& t = ring_trace();
  if (!t.buf) return 0;
  cudaDeviceSynchronize();
  const unsigned k = std::min(std::min(n, t.next), kRingTraceSlots);
  if (k) cudaMemcpy(h_out, t.buf, (size_t)k * 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
  return t.next;
}

// The whole iteration runs as one tiled pass for K = one planar BlockGradient2D (no identity rows),
// prox_g = one Elem1D over all columns with scalar weights (b may be per pixel), prox_f* = one
// Norm2 over the (gx, gy) pair of every voxel with scalar weights, uniform T and Sigma.
bool tile_ring_available(const StencilPlan& plan, const std::vector<ProxDesc>& gd, const std::vector<ProxDesc>& fd,
                         ScaleRef T, ScaleRef S, bool slab) {
  if (!plan.ok || plan.three_d) return false;
  const GradGeom& g = plan.geom;
  if (g.has_id) return false;
  if (g.ny % 4 != 0 || g.plane % 4 != 0 || g.L > 65535u) return false;
  if (T.ptr || S.ptr) return false;
  if (gd.size() != 1 || fd.size() != 1) return false;
  const ProxDesc& pg = gd[0];
  const ProxDesc& pf = fd[0];
  if (pg.kind != kProxElem1D || pg.moreau || pg.index != 0 || pg.dim != 1 || pg.count != g.plane) return false;
  for (int k = 0; k < 7; ++k)
    if (k != 1 && pg.coeffs.ptr[k]) return false;
  if (pg.coeffs.ptr[1] && !aligned16(pg.coeffs.ptr[1])) return false;
  if (pf.kind != kProxNorm2 || pf.moreau || pf.interleaved || pf.index != 0 || pf.dim != 2 ||
      pf.count != g.plane)
    return false;
  for (int k = 0; k < 7; ++k)
    if (pf.coeffs.ptr[k]) return false;
  const uint64_t n_tiles = RingTiles(g).n;
  if (n_tiles == 0 || n_tiles >= (1ull << 31) || !encode_tiled_fn()) return false;
  // the plain and the residual-refresh kernel, with the shared memory they launch with
  for (const bool check : {false, true}) {
    if (cudaFuncSetAttribute(ring_kernel(pg, pf, check, slab), cudaFuncAttributeMaxDynamicSharedMemorySize,
                             kRingSmemBytes) != cudaSuccess) {
      cudaGetLastError();
      return false;
    }
  }
  return true;
}

unsigned tile_ring_grid(const Context* ctx, const StencilPlan& plan) { return RingTiles(plan.geom).grid(ctx); }

unsigned tile_iteration_launch(Context* ctx, const StencilPlan& plan, const ProxDesc& pg, const ProxDesc& pf,
                               const TilePass& p) {
  const unsigned n = ring_launch(ctx, plan.geom, pg, pf, p);
  if (!n) fail(PB_ERR_CUDA, "the one-pass ring kernel could not be launched");
  PB_CHECK_LAUNCH();
  ctx->launches++;
  return p.check ? n : 0;
}

}  // namespace pb
