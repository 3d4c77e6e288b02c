// pb_comm.cu -- NCCL communicator + CUDA-IPC halo blocks for the slab decomposition (pb_comm.cuh).
#include "pb_comm.cuh"

#include <dlfcn.h>
#include <nccl.h>

#include <cstdlib>
#include <cstring>
#include <mutex>

namespace pb {

// device-visible control words of one rank (lives at the start of the IPC block)
struct HaloFlags {
  unsigned x_seq;        // sequence number of the newest x halo written by the RIGHT neighbour
  unsigned y_seq;        // sequence number of the newest y halo written by the LEFT neighbour
  unsigned done_primal;  // local: edge CTAs of the running primal pass that finished
  unsigned done_dual;    // local: same for the dual pass
  int error;             // set by a kernel whose halo wait timed out
  unsigned red_count;    // local: reductions over ranks executed so far (pb_crosssum.cuh)
  int pad[10];
};

namespace {

// ---- lazily loaded NCCL entry points ---------------------------------------------------------------
struct NcclApi {
  ncclResult_t (*GetUniqueId)(ncclUniqueId*);
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int);
  ncclResult_t (*CommDestroy)(ncclComm_t);
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t);
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t);
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
  ncclResult_t (*GroupStart)();
  ncclResult_t (*GroupEnd)();
  const char* (*GetErrorString)(ncclResult_t);
};

NcclApi& nccl() {
  static NcclApi api;
  static std::once_flag once;
  static std::string err;
  std::call_once(once, [] {
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) { err = std::string("cannot load libnccl.so.2: ") + dlerror(); return; }
    auto sym = [&](const char* name) -> void* {
      void* p = dlsym(h, name);
      if (!p && err.empty()) err = std::string("libnccl is missing ") + name;
      return p;
    };
    api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
    api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
    api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
    api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(sym("ncclAllReduce"));
    api.AllGather = reinterpret_cast<decltype(api.AllGather)>(sym("ncclAllGather"));
    api.Send = reinterpret_cast<decltype(api.Send)>(sym("ncclSend"));
    api.Recv = reinterpret_cast<decltype(api.Recv)>(sym("ncclRecv"));
    api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(sym("ncclGroupStart"));
    api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(sym("ncclGroupEnd"));
    api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
  });
  if (!err.empty()) fail(PB_ERR_UNSUPPORTED, "NCCL unavailable: " + err);
  return api;
}

#define PB_NCCL(expr)                                                                       \
  do {                                                                                      \
    ncclResult_t pb_r__ = (expr);                                                           \
    if (pb_r__ != ncclSuccess) {                                                            \
      std::ostringstream pb_ss__;                                                           \
      pb_ss__ << "NCCL error: " << nccl().GetErrorString(pb_r__) << " (" << #expr << " at " \
              << __FILE__ << ":" << __LINE__ << ")";                                        \
      ::pb::fail(PB_ERR_CUDA, pb_ss__.str());                                               \
    }                                                                                       \
  } while (0)

inline ncclComm_t as_comm(void* p) { return static_cast<ncclComm_t>(p); }

// header of the IPC block: HaloFlags | reduce sequence words (offset 256) | reduce slots (offset 512);
// padded so that the float slots behind it stay 16-byte aligned
constexpr size_t kFlagBytes = 2048;
constexpr size_t kRedFlagOff = 256, kRedSlotOff = 512;
constexpr int kRedRanks = 8;         // == kMaxReduceRanks (pb_stencil.cuh)
static_assert(sizeof(HaloFlags) <= kRedFlagOff, "HaloFlags must fit its header");
static_assert(kRedFlagOff + kRedRanks * sizeof(unsigned) <= kRedSlotOff, "reduce flags");
static_assert(kRedSlotOff + 2 * kRedRanks * 4 * sizeof(double) <= kFlagBytes, "reduce slots");

}  // namespace

void Comm::unique_id(void* out128) {
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  ncclUniqueId id;
  PB_NCCL(nccl().GetUniqueId(&id));
  std::memcpy(out128, &id, sizeof(id));
}

Comm::Comm(Context* ctx, int rank, int world, const void* id) : ctx_(ctx), rank_(rank), world_(world) {
  if (world < 1 || rank < 0 || rank >= world) fail(PB_ERR_INVALID, "pb_comm_create: bad rank / world size");
  if (!id) fail(PB_ERR_INVALID, "pb_comm_create: NULL unique id");
  ctx_->bind();
  ncclUniqueId uid;
  std::memcpy(&uid, id, sizeof(uid));
  ncclComm_t c = nullptr;
  PB_NCCL(nccl().CommInitRank(&c, world, uid, rank));
  nccl_ = c;
  const char* mode = std::getenv("PB_HALO");
  p2p_ = !(mode && std::strcmp(mode, "nccl") == 0);
  scratch_.resize(16);
}

Comm::~Comm() {
  cudaSetDevice(ctx_->device);
  cudaStreamSynchronize(ctx_->stream);
  release_halo();
  if (nccl_) nccl().CommDestroy(as_comm(nccl_));
}

void Comm::release_halo() {
  for (int r = 0; r < (int)peer_blocks_.size(); ++r)
    if (r != rank_ && peer_blocks_[r]) cudaIpcCloseMemHandle(peer_blocks_[r]);
  peer_blocks_.clear();
  left_block_ = right_block_ = nullptr;
  if (block_) cudaFree(block_);
  block_ = nullptr;
  flags_ = nullptr;
  x_in_ = y_in_ = nullptr;
  x_ll_ = y_ll_ = nullptr;
  col_floats_ = 0;
}

void Comm::ensure_halo(size_t col_floats) {
  ctx_->bind();
  cudaStream_t s = ctx_->stream;
  // every rank must agree on the size (and on p2p vs staging): checked with one all-reduce
  // (zero variance: sum c = W c and sum c^2 = W c^2 hold on every rank only if all c are equal,
  //  so either every rank throws or none does)
  const double c = static_cast<double>(col_floats);
  double chk[2] = {c, c * c};
  allreduce_sum_host(chk, 2);
  const double mean = chk[0] / world_;
  if (chk[1] / world_ != mean * mean)
    fail(PB_ERR_INVALID, "slab decomposition: ranks disagree on the halo column size (ny * L)");
  x_seq_ = y_seq_ = 0;
  halo_in_ll_ = false;
  if (col_floats == col_floats_ && block_) {
    // same geometry as before: just reset the control words
    PB_CUDA(cudaStreamSynchronize(s));
    barrier();
    PB_CUDA(cudaMemsetAsync(block_, 0, kFlagBytes + 4 * col_floats_ * sizeof(float) + 5 * ll_lines() * sizeof(uint4), s));
    PB_CUDA(cudaStreamSynchronize(s));
    barrier();
    return;
  }
  PB_CUDA(cudaStreamSynchronize(s));
  barrier();                       // nobody still reads a block that is about to be unmapped
  release_halo();
  col_floats_ = col_floats;
  const size_t bytes = kFlagBytes + 4 * col_floats * sizeof(float) + 5 * ll_lines() * sizeof(uint4);
  PB_CUDA(cudaMalloc(&block_, bytes));
  PB_CUDA(cudaMemsetAsync(block_, 0, bytes, s));
  flags_ = static_cast<HaloFlags*>(block_);
  x_in_ = reinterpret_cast<float*>(static_cast<char*>(block_) + kFlagBytes);
  y_in_ = x_in_ + 2 * col_floats;
  x_ll_ = reinterpret_cast<uint4*>(y_in_ + 2 * col_floats);
  y_ll_ = x_ll_ + 2 * ll_lines();
  stage_x_.resize(col_floats);
  stage_y_.resize(col_floats);
  stage_x_.zero(s);
  stage_y_.zero(s);
  PB_CUDA(cudaStreamSynchronize(s));

  // exchange IPC handles (64 bytes per rank) with one all-gather, then map the two neighbours
  int ok = 1;
  if (p2p_ && world_ > 1) {
    cudaIpcMemHandle_t mine;
    std::memset(&mine, 0, sizeof(mine));
    if (cudaIpcGetMemHandle(&mine, block_) != cudaSuccess) { cudaGetLastError(); ok = 0; }
    DeviceBuffer<char> d_all(sizeof(mine) * world_), d_mine(sizeof(mine));
    PB_CUDA(cudaMemcpyAsync(d_mine.data(), &mine, sizeof(mine), cudaMemcpyHostToDevice, s));
    PB_NCCL(nccl().AllGather(d_mine.data(), d_all.data(), sizeof(mine), ncclChar, as_comm(nccl_), s));
    std::vector<cudaIpcMemHandle_t> all(world_);
    PB_CUDA(cudaMemcpyAsync(all.data(), d_all.data(), sizeof(mine) * world_, cudaMemcpyDeviceToHost, s));
    PB_CUDA(cudaStreamSynchronize(s));
    // every rank's block: the neighbours' carry the stencil halos, all of them the residual-sum slots
    peer_blocks_.assign(world_, nullptr);
    peer_blocks_[rank_] = block_;
    for (int r = 0; ok && r < world_; ++r) {
      if (r == rank_) continue;
      if (cudaIpcOpenMemHandle(&peer_blocks_[r], all[r], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
        cudaGetLastError(); peer_blocks_[r] = nullptr; ok = 0;
      }
    }
    if (ok && has_left()) left_block_ = peer_blocks_[rank_ - 1];
    if (ok && has_right()) right_block_ = peer_blocks_[rank_ + 1];
  }
  // p2p only if EVERY rank could map its neighbours; otherwise all ranks fall back to staging
  double okd[1] = {ok ? 0.0 : 1.0};
  allreduce_sum_host(okd, 1);
  if (okd[0] != 0.0 || world_ == 1) {
    if (p2p_ && world_ > 1 && rank_ == 0)
      std::fprintf(stderr, "prost_b200: CUDA IPC halo mapping unavailable, using NCCL send/recv staging\n");
    for (int r = 0; r < (int)peer_blocks_.size(); ++r)
      if (r != rank_ && peer_blocks_[r]) cudaIpcCloseMemHandle(peer_blocks_[r]);
    peer_blocks_.clear();
    left_block_ = right_block_ = nullptr;
    p2p_ = false;
  }
  barrier();
}

float* Comm::x_out(unsigned seq) const {
  if (!has_left()) return nullptr;
  if (!p2p_) return const_cast<float*>(stage_x_.data());
  float* base = reinterpret_cast<float*>(static_cast<char*>(left_block_) + kFlagBytes);
  return base + (seq & 1u) * col_floats_;
}

float* Comm::y_out(unsigned seq) const {
  if (!has_right()) return nullptr;
  if (!p2p_) return const_cast<float*>(stage_y_.data());
  float* base = reinterpret_cast<float*>(static_cast<char*>(right_block_) + kFlagBytes);
  return base + 2 * col_floats_ + (seq & 1u) * col_floats_;
}

uint4* Comm::x_ll_out(unsigned seq) const {
  if (!has_left() || !p2p_ || !left_block_) return nullptr;
  char* base = static_cast<char*>(left_block_) + kFlagBytes + 4 * col_floats_ * sizeof(float);
  return reinterpret_cast<uint4*>(base) + (seq & 1u) * ll_lines();
}

uint4* Comm::y_ll_out(unsigned seq) const {
  if (!has_right() || !p2p_ || !right_block_) return nullptr;
  char* base = static_cast<char*>(right_block_) + kFlagBytes + 4 * col_floats_ * sizeof(float);
  return reinterpret_cast<uint4*>(base) + 2 * ll_lines() + (seq % 3u) * ll_lines();
}

namespace {

// plain column (sequence word protocol of the two-pass kernels) -> flag-in-data lines, local memory only
__global__ void halo_pack_ll_kernel(const float* __restrict__ plain, uint4* __restrict__ ll, unsigned seq,
                                    const unsigned* wait_flag, unsigned groups, int* error) {
  if (wait_flag) {
    unsigned v;
    unsigned long long t0 = 0;
    for (unsigned spins = 0;; ++spins) {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(wait_flag) : "memory");
      if ((int)(v - seq) >= 0) break;
      if ((spins & 1023u) == 1023u) {
        unsigned long long now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        if (t0 == 0) t0 = now;
        else if (now - t0 > 2000000000ull) { if (error) atomicExch(error, 1); break; }
      }
    }
  }
  for (unsigned q = blockIdx.x * blockDim.x + threadIdx.x; q < groups; q += gridDim.x * blockDim.x) {
    const float4 v = __ldcg(reinterpret_cast<const float4*>(plain) + q);
    ll[2 * q] = make_uint4(__float_as_uint(v.x), seq, __float_as_uint(v.y), seq);
    ll[2 * q + 1] = make_uint4(__float_as_uint(v.z), seq, __float_as_uint(v.w), seq);
  }
}

// flag-in-data lines of sequence number `seq` -> plain column (local; the lines are there: the iteration that
// consumed them has completed on this stream)
__global__ void halo_unpack_ll_kernel(const uint4* __restrict__ ll, float* __restrict__ plain, unsigned groups) {
  for (unsigned q = blockIdx.x * blockDim.x + threadIdx.x; q < groups; q += gridDim.x * blockDim.x) {
    const uint4 a = __ldcg(ll + 2 * q), b = __ldcg(ll + 2 * q + 1);
    reinterpret_cast<float4*>(plain)[q] =
        make_float4(__uint_as_float(a.x), __uint_as_float(a.z), __uint_as_float(b.x), __uint_as_float(b.z));
  }
}

}  // namespace

// Primal pass number xs: reads the y columns the left neighbour's dual passes ys / ys-1 delivered, hands column 0
// of the new x to the left.
SlabHalo Comm::primal_halo() {
  const unsigned xs = ++x_seq_, ys = y_seq_;
  SlabHalo h;
  h.has_left = has_left();
  h.has_right = has_right();
  h.in_a = y_slot(ys);
  h.in_b = y_slot(ys - 1);
  h.out = x_out(xs);
  if (p2p_ && h.has_left) {
    h.wait_flag = &flags_->y_seq;
    h.wait_seq = ys;
    h.done_counter = &flags_->done_primal;
    h.signal_flag = &static_cast<HaloFlags*>(left_block_)->x_seq;    // the left neighbour's
    h.signal_seq = xs;
    h.error = &flags_->error;
  }
  return h;
}

// Dual pass number ys: reads the x columns of the right neighbour's primal passes xs / xs-1, hands the last column
// of the new x-component of y to the right.  NCCL staging mode: first the primal pass's x column moves to the left.
SlabHalo Comm::dual_halo() {
  const unsigned xs = x_seq_, ys = ++y_seq_;
  if (!p2p_ && world_ > 1) {
    PB_NCCL(nccl().GroupStart());
    if (has_left()) PB_NCCL(nccl().Send(stage_x_.data(), col_floats_, ncclFloat, rank_ - 1, as_comm(nccl_), ctx_->stream));
    if (has_right()) PB_NCCL(nccl().Recv(x_slot(xs), col_floats_, ncclFloat, rank_ + 1, as_comm(nccl_), ctx_->stream));
    PB_NCCL(nccl().GroupEnd());
  }
  SlabHalo h;
  h.has_left = has_left();
  h.has_right = has_right();
  h.in_a = x_slot(xs);
  h.in_b = x_slot(xs - 1);
  h.out = y_out(ys);
  if (p2p_ && h.has_right) {
    h.wait_flag = &flags_->x_seq;
    h.wait_seq = xs;
    h.done_counter = &flags_->done_dual;
    h.signal_flag = &static_cast<HaloFlags*>(right_block_)->y_seq;   // the right neighbour's
    h.signal_seq = ys;
    h.error = &flags_->error;
  }
  return h;
}

// NCCL staging mode: the dual pass's y column moves to the right.  Peer-to-peer with ring_follows: the received
// plain columns x(x_seq), y(y_seq) are repacked into the local flag-in-data slots once their sequence words arrive.
void Comm::end_two_pass_iteration(bool ring_follows) {
  halo_in_ll_ = false;
  if (!p2p_ && world_ > 1) {
    PB_NCCL(nccl().GroupStart());
    if (has_right()) PB_NCCL(nccl().Send(stage_y_.data(), col_floats_, ncclFloat, rank_ + 1, as_comm(nccl_), ctx_->stream));
    if (has_left()) PB_NCCL(nccl().Recv(y_slot(y_seq_), col_floats_, ncclFloat, rank_ - 1, as_comm(nccl_), ctx_->stream));
    PB_NCCL(nccl().GroupEnd());
  }
  if (!ring_follows || !p2p_ || world_ == 1 || !block_) return;
  const unsigned groups = static_cast<unsigned>(col_floats_ / 4);
  const unsigned grid = std::max(1u, std::min(64u, (groups + 255u) / 256u));
  if (has_right())
    halo_pack_ll_kernel<<<grid, 256, 0, ctx_->stream>>>(x_slot(x_seq_), const_cast<uint4*>(x_ll(x_seq_)), x_seq_,
                                                        &flags_->x_seq, groups, &flags_->error);
  if (has_left())
    halo_pack_ll_kernel<<<grid, 256, 0, ctx_->stream>>>(y_slot(y_seq_), const_cast<uint4*>(y_ll(y_seq_)), y_seq_,
                                                        &flags_->y_seq, groups, &flags_->error);
  PB_CHECK_LAUNCH();
}

// One-pass iteration = primal pass xs and dual pass ys in one launch: the left-edge tiles play the primal pass's
// part of the protocol, the right-edge tiles the dual pass's.
RingHalo Comm::ring_halo() {
  RingHalo h;
  h.has_left = has_left();
  h.has_right = has_right();
  const unsigned ys_in = y_seq_;       // newest y halo (left neighbour's previous iteration)
  const unsigned xs = ++x_seq_, ys = ++y_seq_;
  h.error = &flags_->error;
  if (h.has_left) {
    for (unsigned p = 0; p < 3; ++p) h.yl_ll[p] = y_ll(p);
    for (unsigned p = 0; p < 2; ++p) h.x_out_ll[p] = x_ll_out(p);
    h.y_wait_seq = ys_in;
    h.x_signal_seq = xs;
  }
  if (h.has_right) {
    for (unsigned p = 0; p < 2; ++p) h.xr_ll[p] = x_ll(p);
    for (unsigned p = 0; p < 3; ++p) h.y_out_ll[p] = y_ll_out(p);
    h.x_wait_seq = xs;
    h.y_signal_seq = ys;
  }
  halo_in_ll_ = true;
  return h;
}

Comm::PlainHalo Comm::plain_halo() {
  if (halo_in_ll_ && p2p_ && world_ > 1 && block_) {
    const unsigned groups = static_cast<unsigned>(col_floats_ / 4);
    const unsigned grid = std::max(1u, std::min(64u, (groups + 255u) / 256u));
    auto unpack = [&](const uint4* ll, float* plain) {
      halo_unpack_ll_kernel<<<grid, 256, 0, ctx_->stream>>>(ll, plain, groups);
      PB_CHECK_LAUNCH();
    };
    if (has_right()) {
      unpack(x_ll(x_seq_), x_slot(x_seq_));
      unpack(x_ll(x_seq_ - 1), x_slot(x_seq_ - 1));
    }
    if (has_left()) unpack(y_ll(y_seq_ - 1), y_slot(y_seq_ - 1));
  }
  return {y_slot(y_seq_ - 1), x_slot(x_seq_), x_slot(x_seq_ - 1)};
}

bool Comm::reduce_p2p() const {
  return p2p_ && world_ > 1 && world_ <= kRedRanks && (int)peer_blocks_.size() == world_;
}
const double* Comm::red_in() const {
  return reinterpret_cast<const double*>(static_cast<char*>(block_) + kRedSlotOff);
}
const unsigned* Comm::red_flag_in() const {
  return reinterpret_cast<const unsigned*>(static_cast<char*>(block_) + kRedFlagOff);
}
double* Comm::red_out(int r) const {
  return reinterpret_cast<double*>(static_cast<char*>(peer_blocks_[r]) + kRedSlotOff);
}
unsigned* Comm::red_flag_out(int r) const {
  return reinterpret_cast<unsigned*>(static_cast<char*>(peer_blocks_[r]) + kRedFlagOff);
}

unsigned* Comm::red_count() const { return flags_ ? &flags_->red_count : nullptr; }

CrossSum Comm::cross_sum() const {
  CrossSum c;
  if (!reduce_p2p()) return c;
  c.world = world_;
  c.rank = rank_;
  c.count = red_count();
  c.red_in = red_in();
  c.red_flag_in = red_flag_in();
  for (int r = 0; r < world_; ++r) {
    c.red_out[r] = red_out(r);
    c.red_flag_out[r] = red_flag_out(r);
  }
  c.error = &flags_->error;
  return c;
}

void Comm::allreduce_sum(double* d_buf, size_t n) {
  if (world_ == 1) return;
  PB_NCCL(nccl().AllReduce(d_buf, d_buf, n, ncclDouble, ncclSum, as_comm(nccl_), ctx_->stream));
}

void Comm::allreduce_sum_f32(float* d_buf, size_t n) {
  if (world_ == 1) return;
  PB_NCCL(nccl().AllReduce(d_buf, d_buf, n, ncclFloat, ncclSum, as_comm(nccl_), ctx_->stream));
}

void Comm::allreduce_sum_host(double* h_buf, size_t n) {
  if (world_ == 1) return;
  ctx_->bind();
  if (n > scratch_.size()) scratch_.resize(n);
  scratch_.upload(h_buf, n, ctx_->stream);
  allreduce_sum(scratch_.data(), n);
  scratch_.download(h_buf, n, ctx_->stream);
  PB_CUDA(cudaStreamSynchronize(ctx_->stream));
}

void Comm::exchange_edge_column(const float* d_src, size_t ny, size_t nx, size_t L, bool to_left, float* d_recv) {
  if (world_ == 1) return;
  ctx_->bind();
  cudaStream_t s = ctx_->stream;
  const size_t col = ny * L;
  const int dst = to_left ? rank_ - 1 : rank_ + 1;
  const int src = to_left ? rank_ + 1 : rank_ - 1;
  const bool sends = to_left ? has_left() : has_right();
  const bool receives = to_left ? has_right() : has_left();
  if (sends) {
    // gather the strided column: L rows of ny floats, nx*ny floats apart
    if (edge_send_.size() < col) edge_send_.resize(col);
    const size_t x = to_left ? 0 : nx - 1;
    PB_CUDA(cudaMemcpy2DAsync(edge_send_.data(), ny * sizeof(float), d_src + x * ny, nx * ny * sizeof(float),
                              ny * sizeof(float), L, cudaMemcpyDeviceToDevice, s));
  }
  PB_NCCL(nccl().GroupStart());
  if (sends) PB_NCCL(nccl().Send(edge_send_.data(), col, ncclFloat, dst, as_comm(nccl_), s));
  if (receives) PB_NCCL(nccl().Recv(d_recv, col, ncclFloat, src, as_comm(nccl_), s));
  PB_NCCL(nccl().GroupEnd());
}

void Comm::barrier() {
  double one[1] = {1.0};
  allreduce_sum_host(one, 1);
}

void Comm::check_error() {
  if (!flags_) return;
  int e = 0;
  PB_CUDA(cudaMemcpyAsync(&e, &flags_->error, sizeof(int), cudaMemcpyDeviceToHost, ctx_->stream));
  PB_CUDA(cudaStreamSynchronize(ctx_->stream));
  if (e) fail(PB_ERR_CUDA, "slab decomposition: timed out waiting for a neighbour's stencil halo");
}

}  // namespace pb
