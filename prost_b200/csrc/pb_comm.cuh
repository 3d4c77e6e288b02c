// pb_comm.cuh -- one-process-per-GPU communicator for the slab decomposition (SURVEY.md 8(e)).
//
// The reference is single-GPU (no NCCL/MPI/streams anywhere, SURVEY.md 2a); this layer is what
// lets the fused PDHG passes run on a column slab of a larger grid:
//   * stencil halos travel peer-to-peer: every rank owns a small block of device memory (two
//     ping-pong slots per direction + sequence flags) that its neighbours map through CUDA IPC,
//     and the producing KERNEL stores its edge column straight into the neighbour's slot over
//     NVLink, then publishes a sequence number; the consuming kernel's edge threads spin on that
//     number, so the transfer overlaps the interior of both passes and no copy kernel, no
//     NCCL call and no host synchronisation sits on the iteration path;
//   * the four residual sums are combined with one ncclAllReduce (4 doubles) on the iteration
//     stream at residual_iter boundaries only; every rank then runs the identical step-size
//     state machine on identical bits.
// If CUDA IPC is unavailable (e.g. PB_HALO=nccl, or the mapping fails) the same kernels write the
// edge column to a local staging buffer and the halos move with ncclSend/ncclRecv between the passes.
//
// NCCL is loaded lazily (dlopen libnccl.so.2) so that single-GPU users carry no dependency and a
// process that already loaded torch's bundled NCCL shares that copy.
#pragma once

#include "pb_common.cuh"
#include "pb_crosssum.cuh"

namespace pb {

// Slab decomposition along x (SURVEY.md 8(e)): the local grid is a block of columns of a wider
// image.  The primal pass talks to the LEFT neighbour through its column x = 0 (it needs the
// neighbour's last column of the x-component of y for the divergence and hands over its new
// column 0 of x); the dual pass talks to the RIGHT neighbour through its column x = nx-1 (it needs
// the neighbour's first column of x_new / x_old for the forward difference and hands over its new
// last column of the x-component of y).  `in_a / in_b` are the received columns of the pass's two
// stencil operands (primal: y, y_prev; dual: x_new, x_old), laid out  y + l*ny.  `out` is where the
// outgoing column goes: the neighbour's slot mapped over NVLink (peer-to-peer mode) or a local
// staging buffer (NCCL mode, all flag pointers null).  Comm::primal_halo / dual_halo build it.
struct SlabHalo {
  int has_left = 0, has_right = 0;
  const float* in_a = nullptr;
  const float* in_b = nullptr;
  float* out = nullptr;
  const unsigned* wait_flag = nullptr;   // local sequence word the neighbour publishes to
  unsigned wait_seq = 0;                 // edge threads spin until *wait_flag >= wait_seq (0: no wait)
  unsigned* done_counter = nullptr;      // local: counts finished edge CTAs of this launch
  unsigned n_edge_ctas = 0;
  unsigned* signal_flag = nullptr;       // neighbour's sequence word (peer memory)
  unsigned signal_seq = 0;
  int* error = nullptr;                  // set when a wait times out
};

// Halo descriptor of the one-pass ring kernel (pb_tile.cu) on a slab: ONE launch does the primal and the dual
// step, so it talks to both neighbours.  Its edge columns travel in a flag-in-data layout ("LL", as in NCCL's
// low-latency protocol): every group of four rows is two 16-byte lines {v0, seq, v1, seq} {v2, seq, v3, seq},
// each 8-byte half carrying the sequence number of the iteration that produced it.  The producer's edge warp
// stores the lines straight into the neighbour's memory over NVLink (8-byte halves arrive atomically); the
// consumer's edge warp polls the two lines of ITS rows until all four tags match -- no system-scope fence, no
// edge-tile counter and no separate flag sit between the neighbour's store and this GPU's load (round 1 paid a
// fence.sys on the compute path plus a counter and a flag hop per edge and iteration, profiles/r01_scaling.md).
//   left edge  (tiles of column 0): waits for the left neighbour's newest y.gx column nx-1 (sequence
//              y_wait_seq, produced by its PREVIOUS iteration) row group by row group, computes column 0 and
//              stores its new x column 0 into the left neighbour's x slot tagged x_signal_seq;
//   right edge (tiles owning column nx-1): waits for the right neighbour's new x column 0 of THIS iteration
//              (x_wait_seq; the previous iterate's column is still in the other slot), stores its new y.gx
//              column nx-1 into the right neighbour's y slot tagged y_signal_seq.
// Slot reuse: x has two slots (sequence & 1), y three (sequence % 3: the residual-refresh launch also reads the
// y column before the newest one).  A row group is overwritten only by a thread that has already consumed what
// the overwritten data fed (x: the producer of x(s+2)[r] has seen y(s+1)[r], whose producer had read x(s)[r];
// y(s+3)[r] needs x(s+3)[r], i.e. the neighbour has started launch s+3 and finished every read of launch s+2).
// The left-edge tile column is walked first and the right-edge one in the second wave (pb_tile.cu: decode), so
// in steady state the columns arrive before they are needed.
struct RingHalo {
  int has_left = 0, has_right = 0;
  const uint4* yl_ll[3] = {nullptr, nullptr, nullptr};   // local y slots by (sequence % 3), written by the left rank
  const uint4* xr_ll[2] = {nullptr, nullptr};            // local x slots by (sequence & 1), written by the right rank
  uint4* x_out_ll[2] = {nullptr, nullptr};               // the left neighbour's x slots
  uint4* y_out_ll[3] = {nullptr, nullptr, nullptr};      // the right neighbour's y slots
  unsigned y_wait_seq = 0;             // newest y column from the left (0: none yet)
  unsigned x_wait_seq = 0;             // x column of this iteration from the right
  unsigned x_signal_seq = 0, y_signal_seq = 0;
  int* error = nullptr;                // set when a wait times out
};

struct HaloFlags;   // device-visible control words of one rank (pb_comm.cu)

class Comm {
 public:
  // collective over all ranks; `id` = 128 bytes from unique_id() on rank 0
  Comm(Context* ctx, int rank, int world, const void* id);
  ~Comm();
  static void unique_id(void* out128);

  int rank() const { return rank_; }
  int world() const { return world_; }
  bool p2p() const { return p2p_; }
  bool has_left() const { return rank_ > 0; }
  bool has_right() const { return rank_ + 1 < world_; }
  Context* ctx() const { return ctx_; }

  // collective: (re)allocates the halo block for edge columns of `col_floats` floats and maps the
  // neighbours' blocks; resets the flags and the sequence numbers.  All ranks must pass the same size.
  void ensure_halo(size_t col_floats);
  size_t col_floats() const { return col_floats_; }

  // in-stream sum over ranks of n doubles (device memory, in place)
  void allreduce_sum(double* d_buf, size_t n);
  // in-stream sum over ranks of n floats: the partial K^T r vectors of the row-sharded ADMM (SURVEY.md 8(e))
  void allreduce_sum_f32(float* d_buf, size_t n);
  // host-side conveniences (synchronise the stream)
  void allreduce_sum_host(double* h_buf, size_t n);
  void barrier();

  // collective, for code outside the PDHG passes (the power iteration of the step-size rescaling): one edge
  // column of the planar array d_src (ny x nx x L, idx = y + x*ny + l*nx*ny) moves to a neighbour with grouped
  // ncclSend / ncclRecv on the context stream.  to_left: every rank sends its column 0 to the left neighbour and
  // receives the right neighbour's column 0; otherwise it sends column nx-1 to the right and receives the left
  // neighbour's column nx-1.  d_recv gets ny*L floats laid out y + l*ny (SlabHalo::in_a) and is left untouched on
  // a rank without that neighbour.  Independent of the halo blocks: no sequence number, flag or slot changes, and
  // ensure_halo() need not have run.  All ranks must pass the same ny * L.
  void exchange_edge_column(const float* d_src, size_t ny, size_t nx, size_t L, bool to_left, float* d_recv);

  // --- halo descriptors of the PDHG passes on a slab (pb_pdhg.cu).  All ranks run the same passes, so the pass
  // sequence numbers behind them are identical on every rank.  A two-pass iteration calls primal_halo() before its
  // primal pass, dual_halo() between the passes and end_two_pass_iteration() after the dual pass; a one-pass
  // iteration (ring kernel) calls ring_halo().
  SlabHalo primal_halo();              // next primal pass: newest y columns from the left, x column 0 to the left
  SlabHalo dual_halo();                // next dual pass: this iteration's x columns from the right, y.gx to the right
  // ring_follows: repack the received columns into the flag-in-data slots, where the one-pass iterations read them
  void end_two_pass_iteration(bool ring_follows);
  RingHalo ring_halo();
  // plain halo columns of the iterates y_prev, x and x_prev (current_solution), unpacked from the flag-in-data
  // slots first when a one-pass iteration received the newest ones
  struct PlainHalo { const float* y_prev = nullptr; const float* x = nullptr; const float* x_prev = nullptr; };
  PlainHalo plain_halo();
  // throws if a kernel reported a halo timeout
  void check_error();

  // --- in-kernel sum over ranks (RingFinish, pb_stencil.cuh): every rank's block carries
  // [2][kMaxReduceRanks][4] double slots + one sequence word per writer; all blocks are peer-mapped
  bool reduce_p2p() const;                    // p2p mode, world <= kMaxReduceRanks, every block mapped
  const double* red_in() const;               // local slots
  const unsigned* red_flag_in() const;        // local sequence words
  double* red_out(int r) const;               // rank r's slots (own block for r == rank)
  unsigned* red_flag_out(int r) const;
  unsigned* red_count() const;                // local device counter of executed reductions (pb_crosssum.cuh)
  // descriptor for kernels that sum over ranks themselves (world 1: no-op descriptor)
  struct CrossSum cross_sum() const;

 private:
  void release_halo();
  // local slots: what THIS rank reads
  float* x_slot(unsigned seq) const { return x_in_ + (seq & 1u) * col_floats_; }   // from the right
  float* y_slot(unsigned seq) const { return y_in_ + (seq & 1u) * col_floats_; }   // from the left
  // where THIS rank writes its edge columns: the neighbour's slot (p2p) or the local staging buffer
  float* x_out(unsigned seq) const;   // my column 0 of x      -> left neighbour's x slot
  float* y_out(unsigned seq) const;   // my last column of y.gx -> right neighbour's y slot
  // --- flag-in-data slots of the one-pass ring kernel (RingHalo): two 16-byte lines per four rows
  const uint4* x_ll(unsigned seq) const { return x_ll_ + (seq & 1u) * ll_lines(); }      // local, from the right
  const uint4* y_ll(unsigned seq) const { return y_ll_ + (seq % 3u) * ll_lines(); }      // local, from the left
  uint4* x_ll_out(unsigned seq) const;         // the left neighbour's x slot (p2p only)
  uint4* y_ll_out(unsigned seq) const;         // the right neighbour's y slot
  size_t ll_lines() const { return (col_floats_ + 3) / 4 * 2; }        // 16-byte lines per slot

  Context* ctx_;
  int rank_, world_;
  void* nccl_ = nullptr;               // ncclComm_t
  bool p2p_ = true;
  size_t col_floats_ = 0;
  unsigned x_seq_ = 0, y_seq_ = 0;     // sequence numbers of the newest primal / dual pass
  bool halo_in_ll_ = false;            // the newest halo columns live in the flag-in-data slots only
  // local IPC block: [header: HaloFlags, reduce words and slots | x_in[2][col] | y_in[2][col] | x_ll[2][2 col] |
  // y_ll[3][2 col]]
  void* block_ = nullptr;
  HaloFlags* flags_ = nullptr;
  float* x_in_ = nullptr;
  float* y_in_ = nullptr;
  uint4* x_ll_ = nullptr;              // [2][ll_lines]
  uint4* y_ll_ = nullptr;              // [3][ll_lines]
  void* left_block_ = nullptr;         // neighbours' blocks mapped into this process (p2p)
  void* right_block_ = nullptr;
  std::vector<void*> peer_blocks_;     // every rank's block (own: block_), p2p only
  DeviceBuffer<float> stage_x_, stage_y_;   // staging mode
  DeviceBuffer<float> edge_send_;           // exchange_edge_column: the packed outgoing column
  DeviceBuffer<double> scratch_;
};

}  // namespace pb
