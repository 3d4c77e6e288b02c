// Dense Kronecker products on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a.
//
// kron(K, I_d) x  (block_dense_kron_id.cu:28-58)  is the GEMM  Res (n_out x d) = K (n_out x n_in) X (n_in x d),
// kron(I_d, K) x  (block_id_kron_dense.cu:28-58)  is           Res (d x n_out) = X (d x n_in) K^T,
// with d in the millions and a small factor: 2 n_in n_out flops per (n_in + n_out) floats moved.  From about
// 16 x 32 on the fp32 pipes cannot keep up with HBM (profiles/r02_operators.md: 18 - 36 % of the HBM peak), so
// the products run on the tensor cores with the d-axis as UMMA M:
//
//     D[128 points x n_out] (TMEM, fp32)  =  X_tile[128 x n_in]  *  K^T[n_in x n_out]
//
// * fp32 parity through the 3 x TF32 split: every operand is written to shared memory as hi = tf32(x) (round to
//   nearest) and lo = x - hi (exact); D = X_hi K_hi + X_lo K_hi + X_hi K_lo, accumulated in fp32 in TMEM.  The
//   dropped X_lo K_lo term and the truncation of lo are ~2^-21 relative to sum |x||k| per product.
// * the X tile is split by the threads on its way from registers to shared memory, so no TMA: 128-bit global loads
//   of the NEXT tile are in flight while the tensor core works on the current one and the previous tile's
//   accumulator (the other half of the TMEM allocation) is drained to HBM.
// * shared-memory operand layouts are the canonical no-swizzle ("interleave") K-major UMMA layouts: 8 x 16-byte core
//   matrices, for the X tile (A operand) and for the factor (B operand [n_out x n_in], split and laid out once on
//   the host).
//   Descriptor bit fields: cute/arch/mma_sm100_desc.hpp (SmemDescriptor, InstrDescriptor) of the CUTLASS headers in
//   this image; the code below only uses the PTX instructions.
// * one persistent CTA per SM (16 worker warps + one MMA warp), tiles of 128 points round-robin.
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <vector>

#include <cuda.h>

#include "pb_common.cuh"
#include "pb_linop.cuh"

namespace pb {

namespace {

constexpr int kTcWorkerWarps = 16;
constexpr int kTcWorkers = kTcWorkerWarps * 32;
constexpr int kTcThreads = kTcWorkers + 32;     // + the MMA warp
constexpr int kTcUnits = 4;               // 16-byte operand units per worker and tile: 128 points * 16 chunks / 512
constexpr int kTcPoints = 128;            // UMMA M
constexpr uint32_t kTcMaxIn = 64;         // padded factor columns (UMMA K total): kTcUnits operand units per worker
constexpr uint32_t kTcMaxOut = 256;       // padded factor rows (UMMA N)
constexpr size_t kTcMaxSmem = 220 * 1024;

__device__ __forceinline__ uint32_t tc_smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void tc_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(tc_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void tc_mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc_smem_u32(bar)) : "memory");
}
// barrier 1: the worker warps only
__device__ __forceinline__ void tc_worker_barrier() { asm volatile("bar.sync 1, %0;" ::"n"(16 * 32) : "memory"); }
__device__ __forceinline__ void tc_mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n selp.u32 %0, 1, 0, p;\n}"
        : "=r"(done) : "r"(tc_smem_u32(bar)), "r"(parity), "r"(1000000u) : "memory");
  }
}
// shared-memory matrix descriptor, no swizzle: start address, leading / stride byte offsets (16-byte units),
// descriptor version 1 (Blackwell) in bits 46-47, layout type 0 in bits 61-63
__device__ __forceinline__ uint64_t tc_smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return static_cast<uint64_t>((addr & 0x3FFFFu) >> 4) | (static_cast<uint64_t>(lbo_bytes >> 4) << 16) |
         (static_cast<uint64_t>(sbo_bytes >> 4) << 32) | (1ull << 46);
}
// D (+)= A B, kind::tf32, one CTA; issued by one thread
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n"
      " tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tc_smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_ld8(uint32_t taddr, float (&v)[8]) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tc_ld4(uint32_t taddr, float (&v)[4]) {
  uint32_t r[4];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 4; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, "
      "[%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
// nearest tf32 (10 mantissa bits), ties away from zero -- what cvt.rna.tf32.f32 returns for finite inputs and
// infinities, in two integer instructions (the PTX instruction expands to four with its NaN handling)
__device__ __forceinline__ float tc_round_tf32(float x) {
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
}

struct KronTcArgs {
  float* res;
  const float* rhs;
  const uint4* f_hi;          // factor, K-major B layout, padded: n_out_pad x k_pad floats
  const uint4* f_lo;
  uint32_t n_out, n_in, n_out_pad, k_pad;
  size_t d;
  uint32_t tmem_cols;
  uint32_t tma_out;           // kron(K, I): results leave as one TMA tensor store per warp (32 points x its columns)
  uint32_t stage_out;         // kron(I, K): results leave through a shared-memory tile (n_out % 4 == 0, n_out <= 64)
  const int* skip;
};

// IDFIRST = false: kron(K, I_d)   rhs[i*d + p],     res[o*d + p]
// IDFIRST = true : kron(I_d, K)   rhs[p*n_in + i],  res[p*n_out + o]
//
// Both operands are K-major in shared memory: core matrix = 8 rows (points / factor rows) x 16 bytes (4 k), rows 16
// bytes apart; the two 16-byte k-chunks of a k-step (UMMA K = 8 for tf32) are 128 bytes apart (leading byte offset),
// groups of 8 rows k_pad * 32 bytes apart (stride byte offset).  Element (row r, k):
//     (r / 8) * k_pad * 32 + (k / 4) * 128 + (r % 8) * 16 + (k % 4) * 4.
// A worker thread owns whole 16-byte (row, k-chunk) units with the 8 rows of a core matrix on 8 neighbouring lanes,
// so its 128-bit shared-memory stores are conflict-free:
//   kron(I, K): X is k-contiguous, a unit is one 128-bit load;
//   kron(K, I): X is point-contiguous, a unit is four 32-bit loads (rows k .. k + 3 of X at one point; a warp reads
//               128 contiguous bytes of each row).
//
// Roles: 16 worker warps (load -> split -> shared memory; TMEM -> HBM) and one MMA warp.  Per operand / accumulator
// buffer b (two of each): workers arrive on full[b] after writing tile j's operands, the MMA warp waits for it, issues
// the 3 * k_pad / 8 MMAs and commits them to done[b]; every worker waits for that before it drains tile j, which is
// also what allows it to overwrite buffer b with tile j + 2.  No CTA-wide barrier inside the loop.
template <bool IDFIRST, bool SET>
__global__ void __launch_bounds__(kTcThreads, 1) kron_tc_kernel(const KronTcArgs a,
                                                                const __grid_constant__ CUtensorMap out_map) {
  if (a.skip && *a.skip) return;
  extern __shared__ __align__(128) uint8_t tc_smem[];
  const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t ko_count = a.k_pad >> 3;                 // k-steps of 8 (one tf32 UMMA each)
  const uint32_t kc_count = a.k_pad >> 2;                 // 16-byte k-chunks per row
  const uint32_t sbo = a.k_pad * 32u;
  const uint32_t xb = ko_count * 4096u;                   // one X operand buffer: 128 points x k_pad floats
  const uint32_t fb = a.n_out_pad * a.k_pad * 4u;         // one factor operand
  uint8_t* const x_hi0 = tc_smem;                         // [buf][hi, lo]
  uint8_t* const f_hi = tc_smem + 4 * xb;
  uint8_t* const f_lo = f_hi + fb;
  uint64_t* const full = reinterpret_cast<uint64_t*>(f_lo + fb);
  uint64_t* const done = full + 2;                        // one per accumulator
  uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(full + 6);

  for (uint32_t i = tid; i < fb / 16; i += kTcThreads) {
    reinterpret_cast<uint4*>(f_hi)[i] = __ldg(a.f_hi + i);
    reinterpret_cast<uint4*>(f_lo)[i] = __ldg(a.f_lo + i);
  }
  if (tid == 0) {
    tc_mbar_init(&full[0], kTcWorkerWarps);
    tc_mbar_init(&full[1], kTcWorkerWarps);
    tc_mbar_init(&done[0], 1);
    tc_mbar_init(&done[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem_u32(tmem_slot)),
                 "r"(a.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
  const size_t tiles = (a.d + kTcPoints - 1) / kTcPoints;
  const size_t stride = gridDim.x;

  if (warp == kTcWorkerWarps) {
    // ---- MMA warp ----
    // instruction descriptor: D fp32 (bits 4-5 = 1), A / B tf32 (bits 7-9, 10-12 = 2), A and B K-major (bits 15, 16 =
    // 0), N >> 3 in bits 17-22, M >> 4 in bits 24-28
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((a.n_out_pad >> 3) << 17) |
                           ((uint32_t)(kTcPoints >> 4) << 24);
    const uint64_t db_hi0 = tc_smem_desc(tc_smem_u32(f_hi), 128u, sbo), db_lo0 = tc_smem_desc(tc_smem_u32(f_lo), 128u, sbo);
    uint32_t j = 0;
    for (size_t t = blockIdx.x; t < tiles; t += stride, ++j) {
      const uint32_t buf = j & 1;
      tc_mbar_wait(&full[buf], (j >> 1) & 1);
      tc_fence_after();
      if (lane == 0) {
        const uint32_t xh = tc_smem_u32(x_hi0 + buf * 2 * xb);
        const uint64_t da_hi0 = tc_smem_desc(xh, 128u, sbo), da_lo0 = tc_smem_desc(xh + xb, 128u, sbo);
        const uint32_t dst = tmem + buf * a.n_out_pad;
        for (uint32_t ko = 0; ko < ko_count; ++ko) {
          const uint64_t step = ko * 16u;                      // 256 bytes per k-step, in 16-byte units
          tc_mma_tf32(dst, da_hi0 + step, db_hi0 + step, idesc, ko > 0);
          tc_mma_tf32(dst, da_lo0 + step, db_hi0 + step, idesc, 1u);
          tc_mma_tf32(dst, da_hi0 + step, db_lo0 + step, idesc, 1u);
        }
        tc_commit(&done[buf]);
      }
      __syncwarp();
    }
  } else {
    // ---- worker warps ----
    // this thread's units: shared-memory offset, source pointer for tile 0, point within the tile, valid k count
    uint32_t soff[kTcUnits], upt[kTcUnits], ukn[kTcUnits];
    const float* gsrc[kTcUnits];
#pragma unroll
    for (uint32_t it = 0; it < kTcUnits; ++it) {
      const uint32_t u = it * kTcWorkers + tid;
      uint32_t pt, kc;
      if (!IDFIRST) {
        pt = u & 127u;
        kc = u >> 7;
      } else {
        const uint32_t rest = u >> 3, g = rest / kc_count;
        kc = rest - g * kc_count;
        pt = g * 8 + (u & 7u);
      }
      const bool ok = u < 128u * kc_count;
      soff[it] = (pt >> 3) * sbo + kc * 128u + (pt & 7u) * 16u;
      upt[it] = ok ? pt : 0xffffffffu;
      ukn[it] = (ok && 4 * kc < a.n_in) ? min(4u, a.n_in - 4 * kc) : 0u;
      gsrc[it] = IDFIRST ? a.rhs + (size_t)pt * a.n_in + 4 * kc : a.rhs + (size_t)(4 * kc) * a.d + pt;
    }
    float4 stage[kTcUnits];

    const size_t dd = a.d, dd2 = 2 * dd, dd3 = 3 * dd;
    auto load_tile = [&](float4 (&st)[kTcUnits], size_t t) {
      const size_t p0 = t * kTcPoints;
      const size_t base = IDFIRST ? p0 * a.n_in : p0;
      const bool whole = p0 + kTcPoints <= dd;
#pragma unroll
      for (uint32_t it = 0; it < kTcUnits; ++it) {
        st[it] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (upt[it] == 0xffffffffu) continue;
        const float* src = gsrc[it] + base;
        if (IDFIRST) {
          if (ukn[it] > 0 && (whole || p0 + upt[it] < dd)) st[it] = __ldcs(reinterpret_cast<const float4*>(src));
        } else if (whole && ukn[it] == 4) {
          st[it].x = __ldcs(src);
          st[it].y = __ldcs(src + dd);
          st[it].z = __ldcs(src + dd2);
          st[it].w = __ldcs(src + dd3);
        } else if (p0 + upt[it] < dd) {
          if (ukn[it] > 0) st[it].x = __ldcs(src);
          if (ukn[it] > 1) st[it].y = __ldcs(src + dd);
          if (ukn[it] > 2) st[it].z = __ldcs(src + 2 * dd);
          if (ukn[it] > 3) st[it].w = __ldcs(src + 3 * dd);
        }
      }
    };
    auto store_tile = [&](const float4 (&st)[kTcUnits], uint32_t buf) {
      uint8_t* const hi = x_hi0 + buf * 2 * xb;
      uint8_t* const lo = hi + xb;
#pragma unroll
      for (uint32_t it = 0; it < kTcUnits; ++it) {
        if (upt[it] != 0xffffffffu) {
          const float4 v = st[it];
          float4 h, l;
          h.x = tc_round_tf32(v.x); h.y = tc_round_tf32(v.y); h.z = tc_round_tf32(v.z); h.w = tc_round_tf32(v.w);
          l.x = v.x - h.x; l.y = v.y - h.y; l.z = v.z - h.z; l.w = v.w - h.w;
          *reinterpret_cast<float4*>(hi + soff[it]) = h;
          *reinterpret_cast<float4*>(lo + soff[it]) = l;
        }
      }
    };
    // Warp w reads TMEM lanes 32 (w % 4) ..; the four warps of a lane quarter split the columns.
    const uint32_t lb = warp & 3, cols = a.n_out_pad >> 2, c_begin = (warp >> 2) * cols;
    const uint32_t row = 32 * lb + lane;                              // this thread's point within a tile
    const uint32_t nvalid = c_begin < a.n_out ? min(cols, a.n_out - c_begin) : 0u;   // real columns of this warp
    // kron(K, I): column c of the accumulator is row c of res (a warp stores 128 contiguous bytes per column)
    float* const out_col0 = IDFIRST ? a.res + (size_t)row * a.n_out + c_begin : a.res + (size_t)c_begin * dd + row;
    // kron(I, K), staged: the tile's 128 x n_out results are one contiguous block of res.  The accumulator rows go to
    // a padded shared-memory tile (row stride odd in 16-byte units: conflict-free 128-bit stores) and leave it as
    // 512 contiguous bytes per warp store; a lane-per-row store would touch 32 lines per instruction.
    const bool staged = IDFIRST && a.stage_out;
    const uint32_t q_per_row = a.n_out >> 2, stride16 = q_per_row | 1u;
    uint8_t* const stg = reinterpret_cast<uint8_t*>(full) + 128;
    uint32_t cp_soff[kTcUnits];
    if (staged) {
#pragma unroll
      for (uint32_t it = 0; it < kTcUnits; ++it) {
        const uint32_t u = it * kTcWorkers + tid, r = u / q_per_row;
        cp_soff[it] = (r * stride16 + (u - r * q_per_row)) * 16u;
      }
    }
    // columns [c, c + 4) of this thread's accumulator row -> HBM (dst: column c of this thread's point)
    auto put4 = [&](const float* v, uint32_t c, float* dst) {
      if (!IDFIRST) {
        if (c + 4 <= c_begin + nvalid) {
          if (SET) { __stcs(dst, v[0]); __stcs(dst + dd, v[1]); __stcs(dst + dd2, v[2]); __stcs(dst + dd3, v[3]); }
          else { dst[0] += v[0]; dst[dd] += v[1]; dst[dd2] += v[2]; dst[dd3] += v[3]; }
        } else {
#pragma unroll
          for (uint32_t q = 0; q < 4; ++q)
            if (c + q < c_begin + nvalid) { if (SET) __stcs(dst + q * dd, v[q]); else dst[q * dd] += v[q]; }
        }
      } else if (c < c_begin + nvalid) {
        if ((a.n_out & 3u) == 0) {
          float4 o = make_float4(v[0], v[1], v[2], v[3]);
          float4* d4 = reinterpret_cast<float4*>(dst);
          if (!SET) { const float4 r = *d4; o.x += r.x; o.y += r.y; o.z += r.z; o.w += r.w; }
          __stcs(d4, o);
        } else {
#pragma unroll
          for (uint32_t q = 0; q < 4; ++q)
            if (c + q < c_begin + nvalid) { if (SET) dst[q] = v[q]; else dst[q] += v[q]; }
        }
      }
    };
    // accumulator of tile t (TMEM half `acc`) -> HBM
    auto drain = [&](size_t t, uint32_t acc, uint32_t parity) {
      tc_mbar_wait(&done[acc], parity);
      tc_fence_after();
      const size_t p0 = t * kTcPoints;
      const bool live = p0 + row < dd;
      const uint32_t taddr = tmem + ((32u * lb) << 16) + acc * a.n_out_pad;
      if (!IDFIRST && a.tma_out) {
        // kron(K, I) through TMA: the warp's 32 points x cols accumulators go to its own [cols][32] shared-memory tile
        // (128 contiguous bytes per column: conflict-free) and leave as ONE tensor store (or add-reduction) instead of
        // cols store instructions per thread with their 64-bit address arithmetic; out-of-range points / columns are
        // clipped by the tensor map
        float* const tile = reinterpret_cast<float*>(stg + warp * (cols * 128u));
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // previous store has read it
        __syncwarp();
        uint32_t c = 0;
        for (; c + 16 <= cols; c += 16) {
          float v[16];
          tc_ld16(taddr + c_begin + c, v);
#pragma unroll
          for (uint32_t q = 0; q < 16; ++q) tile[(c + q) * 32 + lane] = v[q];
        }
        if (c + 8 <= cols) {
          float v[8];
          tc_ld8(taddr + c_begin + c, v);
#pragma unroll
          for (uint32_t q = 0; q < 8; ++q) tile[(c + q) * 32 + lane] = v[q];
          c += 8;
        }
        if (c < cols) {
          float v[4];
          tc_ld4(taddr + c_begin + c, v);
#pragma unroll
          for (uint32_t q = 0; q < 4; ++q) tile[(c + q) * 32 + lane] = v[q];
        }
        tc_fence_before();
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
          const uint64_t map = reinterpret_cast<uint64_t>(&out_map);
          const uint32_t src = tc_smem_u32(tile);
          const int x = (int)(p0 + 32 * lb), y = (int)c_begin;
          if (SET)
            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];"
                         ::"l"(map), "r"(x), "r"(y), "r"(src) : "memory");
          else
            asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%1, %2}], [%3];"
                         ::"l"(map), "r"(x), "r"(y), "r"(src) : "memory");
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        return;
      }
      float* dst = staged ? reinterpret_cast<float*>(stg + (row * stride16 + (c_begin >> 2)) * 16u)
                          : out_col0 + (IDFIRST ? p0 * a.n_out : p0);
      const size_t cstep = (IDFIRST || staged) ? 1 : dd;              // distance between columns at dst
      uint32_t c = c_begin;
      const uint32_t c_end = c_begin + cols;
      for (; c + 16 <= c_end; c += 16) {
        float v[16];
        tc_ld16(taddr + c, v);
        if (staged) {
#pragma unroll
          for (uint32_t q = 0; q < 16; q += 4)
            if (c + q < c_begin + nvalid)
              *reinterpret_cast<float4*>(dst + q) = make_float4(v[q], v[q + 1], v[q + 2], v[q + 3]);
        } else if (live) {
#pragma unroll
          for (uint32_t q = 0; q < 16; q += 4) put4(v + q, c + q, dst + q * cstep);
        }
        dst += 16 * cstep;
        __syncwarp();          // the TMEM loads are warp-collective
      }
      if (c + 8 <= c_end) {
        float v[8];
        tc_ld8(taddr + c, v);
        if (staged) {
#pragma unroll
          for (uint32_t q = 0; q < 8; q += 4)
            if (c + q < c_begin + nvalid)
              *reinterpret_cast<float4*>(dst + q) = make_float4(v[q], v[q + 1], v[q + 2], v[q + 3]);
        } else if (live) {
          put4(v, c, dst);
          put4(v + 4, c + 4, dst + 4 * cstep);
        }
        dst += 8 * cstep;
        __syncwarp();
        c += 8;
      }
      if (c < c_end) {
        float v[4];
        tc_ld4(taddr + c, v);
        if (staged) {
          if (c < c_begin + nvalid) *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
        } else if (live) {
          put4(v, c, dst);
        }
        __syncwarp();
      }
      tc_fence_before();
      if (staged) {
        tc_worker_barrier();                                           // the tile is complete in shared memory
        const size_t rows_valid = min((size_t)kTcPoints, dd - p0);
        const uint32_t units = (uint32_t)rows_valid * q_per_row;
        float4* const out = reinterpret_cast<float4*>(a.res + p0 * a.n_out);
#pragma unroll
        for (uint32_t it = 0; it < kTcUnits; ++it) {
          const uint32_t u = it * kTcWorkers + tid;
          if (u < units) {
            float4 o = *reinterpret_cast<const float4*>(stg + cp_soff[it]);
            if (!SET) { const float4 r = out[u]; o.x += r.x; o.y += r.y; o.z += r.z; o.w += r.w; }
            __stcs(out + u, o);
          }
        }
        tc_worker_barrier();                                           // before the next tile overwrites it
      }
    };

    if (blockIdx.x < tiles) load_tile(stage, blockIdx.x);
    // Tile j of this CTA (tile t = blockIdx.x + j * stride): operand buffer and accumulator j % 2.  It is drained in
    // iteration j + 1, after tile j + 1's operands were written, so that its MMAs (and their completion latency) are
    // off the workers' critical path; the iteration past the last tile only drains.
    uint32_t j = 0;
    for (size_t t = blockIdx.x;; t += stride, ++j) {
      if (t < tiles) {
        const uint32_t buf = j & 1;
        // operand buffer `buf` was last read by the MMAs of tile j - 2: this thread waited for them when it drained
        // tile j - 2 in the previous iteration
        store_tile(stage, buf);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        tc_fence_before();
        __syncwarp();
        if (lane == 0) tc_mbar_arrive(&full[buf]);
        if (t + stride < tiles) load_tile(stage, t + stride);
      }
      if (j >= 1) drain(t - stride, (j - 1) & 1, ((j - 1) >> 1) & 1);
      if (t >= tiles) break;
    }
    if (!IDFIRST && a.tma_out && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(a.tmem_cols) : "memory");
  }
}

inline float host_round_tf32(float x) {     // cvt.rna.tf32.f32: nearest, ties away from zero, 10 mantissa bits
  uint32_t b;
  std::memcpy(&b, &x, 4);
  if ((b & 0x7f800000u) == 0x7f800000u) return x;
  b = (b + 0x1000u) & 0xffffe000u;
  float r;
  std::memcpy(&r, &b, 4);
  return r;
}

}  // namespace

bool KronTensorCore::supported(bool id_first, uint32_t n_out, uint32_t n_in, size_t d, const float* res,
                               const float* rhs) {
  if (d == 0 || n_out == 0 || n_in == 0) return false;
  const uint32_t k_pad = (n_in + 7u) & ~7u, n_pad = (n_out + 15u) & ~15u;
  if (k_pad > kTcMaxIn || n_pad > kTcMaxOut) return false;
  if ((size_t)n_in * n_out < 512) return false;            // small factors: the fp32 kernels are at the HBM bound
  if (id_first && ((reinterpret_cast<uintptr_t>(res) | reinterpret_cast<uintptr_t>(rhs)) & 15u) != 0) return false;
  if (id_first && n_in % 4 != 0) return false;      // 128-bit loads of the k-contiguous rows
  return smem_bytes(id_first, n_out, n_pad, k_pad) <= kTcMaxSmem;
}

static bool stages_output(bool id_first, uint32_t n_out) { return id_first && n_out % 4 == 0 && n_out <= 64; }

typedef CUresult (*TcEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static TcEncodeTiledFn tc_encode_fn() {
  static TcEncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    cudaGetLastError();
    return reinterpret_cast<TcEncodeTiledFn>(p);
  }();
  return fn;
}
// res of kron(K, I) as a 2-D tensor [n_out rows][d points]; box = 32 points x the columns of one warp.  false: the
// results leave through per-thread stores instead
static bool tc_out_map(float* res, size_t d, uint32_t n_out, uint32_t cols, CUtensorMap& m) {
  if (d % 4 != 0 || (reinterpret_cast<uintptr_t>(res) & 15u) != 0 || cols > 256 || d >= (1ull << 31)) return false;
  TcEncodeTiledFn enc = tc_encode_fn();
  if (!enc) return false;
  const cuuint64_t dims[2] = {(cuuint64_t)d, (cuuint64_t)n_out};
  const cuuint64_t strides[1] = {(cuuint64_t)d * 4};
  const cuuint32_t box[2] = {32, cols};
  const cuuint32_t estr[2] = {1, 1};
  return enc(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, res, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

size_t KronTensorCore::smem_bytes(bool id_first, uint32_t n_out, uint32_t n_pad, uint32_t k_pad) {
  // output staging: kron(I, K) a padded 128 x n_out tile, kron(K, I) [n_pad][128] for the per-warp tensor stores
  const size_t staging = stages_output(id_first, n_out) ? (size_t)kTcPoints * ((n_out / 4) | 1u) * 16
                         : !id_first ? (size_t)n_pad * kTcPoints * 4 : 0;
  return 4 * (size_t)(k_pad / 8) * 4096 + 2 * (size_t)n_pad * k_pad * 4 + 128 + staging;
}

// K(o, i) = k[o * so + i * si]  ->  hi / lo parts in the K-major no-swizzle operand layout, zero padded
void KronTensorCore::pack(Context* ctx, const float* k, uint32_t n_out, uint32_t n_in, uint32_t so, uint32_t si,
                          Packed& out) {
  out.n_pad = (n_out + 15u) & ~15u;
  out.k_pad = (n_in + 7u) & ~7u;
  std::vector<float> hi((size_t)out.n_pad * out.k_pad, 0.f), lo(hi.size(), 0.f);
  for (uint32_t r = 0; r < n_out; ++r)
    for (uint32_t c = 0; c < n_in; ++c) {
      const size_t byte = (size_t)(r / 8) * out.k_pad * 32 + (size_t)(c / 4) * 128 + (r % 8) * 16 + (c % 4) * 4;
      const float v = k[(size_t)r * so + (size_t)c * si];
      hi[byte / 4] = host_round_tf32(v);
      lo[byte / 4] = v - hi[byte / 4];
    }
  out.hi.assign(hi, ctx->stream);
  out.lo.assign(lo, ctx->stream);
  out.ready = true;
}

void KronTensorCore::launch(Context* ctx, bool id_first, const Packed& f, float* res, const float* rhs, uint32_t n_out,
                            uint32_t n_in, size_t d, bool set) {
  KronTcArgs a;
  a.res = res;
  a.rhs = rhs;
  a.f_hi = reinterpret_cast<const uint4*>(f.hi.data());
  a.f_lo = reinterpret_cast<const uint4*>(f.lo.data());
  a.n_out = n_out;
  a.n_in = n_in;
  a.n_out_pad = f.n_pad;
  a.k_pad = f.k_pad;
  a.d = d;
  uint32_t cols = 32;                                        // two accumulators, a power of two >= 32 columns
  while (cols < 2 * f.n_pad) cols *= 2;
  a.tmem_cols = cols;
  a.skip = ctx->skip_flag;
  const size_t smem = smem_bytes(id_first, n_out, f.n_pad, f.k_pad);
  a.stage_out = stages_output(id_first, n_out) ? 1u : 0u;
  CUtensorMap out_map;
  std::memset(&out_map, 0, sizeof(out_map));
  a.tma_out = (!id_first && tc_out_map(res, d, n_out, f.n_pad / 4, out_map)) ? 1u : 0u;
  const size_t tiles = (d + kTcPoints - 1) / kTcPoints;
  const unsigned grid = (unsigned)std::min<size_t>(tiles, (size_t)ctx->num_sms);
#define PB_TC(I, S)                                                                                          \
  do {                                                                                                       \
    PB_CUDA(cudaFuncSetAttribute(kron_tc_kernel<I, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    kron_tc_kernel<I, S><<<grid, kTcThreads, smem, ctx->stream>>>(a, out_map);                               \
  } while (0)
  if (id_first) { if (set) PB_TC(true, true); else PB_TC(true, false); }
  else { if (set) PB_TC(false, true); else PB_TC(false, false); }
#undef PB_TC
}

}  // namespace pb
