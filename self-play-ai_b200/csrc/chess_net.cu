// chess_net.cu — the chess policy/value network on tcgen05 tensor cores (sm_100a).
//
// Replaces Net::forward of src/model/chess.rs:75-83 (torso src/model/mod.rs:152-184) and the tensor part of Model::predict
// (src/model/mod.rs:60-67).  Unlike the 4 x 64 nets (evaluator_umma.cu), a batch of chess activations does not fit in shared
// memory (256 channels x 64 cells x 2 B = 32 KB per position), so the network runs layer by layer over the whole leaf
// batch: one launch of k_conv per convolution, activations in HBM/L2 between layers (bf16), all arithmetic f32-accumulated.
//
// Activation layout ("planar, 81-row boards"): a position is 9 x 9 = 81 rows (8 x 8 cells + one zero pad column + one
// zero pad row, the pad row shared with the next position), so a 3x3 tap (dy,dx) is the constant row offset dy*9+dx and
// the pads supply the conv's zero padding.  Channels are split into chunks of 8 (16 bytes); HBM holds one plane per
// chunk, [chunk][row][8 ch] — a tile of rows of one chunk is one contiguous run (one cp.async.bulk) and lands in shared
// memory as the K-major no-swizzle UMMA operand layout (8-row core matrices of 128 contiguous bytes at ANY row offset, so a
// tap shift is just the descriptor's start address: verified by tools/umma_probe.cu).
//
// k_conv<KC32, TAPS, N, EPI>: persistent CTAs, one M tile at a time, implicit GEMM M = 128, N = 256 (80 for the last policy
// conv), K = TAPS x KC32 x 32.  An M tile is 16 board rows of 8 cells: the A descriptor strides 9 layout rows (144 B) between
// its 8-row core matrices, so the zero pad column never enters the MMA (8/9 of the tile rows are real cells).
//   warp 0      producer: A tile (169 layout rows incl. halo, all input channels, loaded ONCE per tile and reused by the 9
//               taps) and the weight stream (16 KB stages of 32 input channels x 256 outputs through an 8-deep ring = 2,000
//               cycles of cover for the L2 latency), cp.async.bulk + mbarrier complete_tx.  CTAs run in PAIRS (clusters of
//               2) on different tiles with the same weights: each loads half of every stage and multicasts it to both.
//   warp 1      MMA issuer: tcgen05.mma.cta_group::1.kind::f16 M = 128, N = 256, K = 16: 128 cycles each = the tensor
//               pipe's rate, 144 per tile; accumulators in TMEM, 2 x 256 columns (double buffered)
//   warps 2-5   epilogue: tcgen05.ld -> + bias (+ skip) -> ReLU -> bf16 -> HBM, or f32 logits; pad cells are never written
//               (they are zero from the allocation on and supply the conv's zero padding)
// The K loop runs channel-group major (8 groups of 32 input channels, 9 taps each), so the A tile is 8 independent
// sub-buffers: group g of the NEXT tile is loaded as soon as the 9 taps of group g of this tile have been read — the A
// load is double-buffered at 1/8 granularity inside ONE 85 KB buffer, which leaves 128 KB for the weight ring.  The
// epilogue of tile i overlaps the MMAs of tile i+1.
// Algorithmic bytes per tile-layer: A 85 KB + weights 1,152 KB (L2-resident, 1.2 MB per layer) in, 57 KB out, against
// 134 MFLOP of real cells (151 MFLOP issued): the kernel is tensor-bound (18.4 k cycles of MMA per tile) as long as L2
// sustains 64 B/clk/SM of weight traffic.
#include <cuda_bf16.h>

#include <cstring>

#include "bf16.cuh"
#include "chess_engine.hpp"
#include "chess_net.cuh"
#include "umma_ptx.cuh"

namespace spb {
namespace chess {

using namespace spb::umma;

constexpr int BOARD_ROWS = 81;        // layout rows of one position: 9 board rows (8 + the shared zero row) x 9 cells (8 + the zero column)
constexpr int LEAD = 16;              // zero rows in front of the first position (taps reach back 10 rows)
// An M tile is 16 BOARD ROWS of 8 real cells: the A descriptor's stride between 8-row core matrices (SBO) is 9 layout rows
// (144 bytes), so the zero pad COLUMN never enters the MMA — 8 of every 9 tile rows are real cells (the 9th board row of a
// position, its zero pad row, still does): 89 % useful rows instead of 79 % with 128 consecutive layout rows per tile.
constexpr int TILE_BROWS = 16;                    // board rows per tile
constexpr int TILE_SPAN = TILE_BROWS * 9;         // layout rows one tile spans: 144
constexpr int QA = 16 + (TILE_BROWS - 1) * 9 + 8 + 10;   // rows of an A tile in shared memory: 16 halo + 143 + 10 halo = 169
#ifndef SPB_CHESS_NSTAGE
#define SPB_CHESS_NSTAGE 8
#endif
constexpr int NSTAGE = SPB_CHESS_NSTAGE;   // weight ring depth
constexpr int CONV_THREADS = 192;
constexpr int IN_CHUNKS = 4;          // stem input: 19 planes padded to 32 channels

__host__ __device__ constexpr uint32_t tiles_for(uint32_t boards) { return (boards * 9u + TILE_BROWS - 1u) / TILE_BROWS; }
// + one tile: the second CTA of a pair runs a dummy tile when the number of tiles is odd
__host__ __device__ constexpr size_t plane_rows_for(uint32_t max_boards) { return (size_t)LEAD + (size_t)(tiles_for(max_boards) + 1) * TILE_SPAN + 64; }

// ---- CTA pairs: the two CTAs of a cluster work on different M tiles with the SAME weights, so each loads half of every
// weight stage and multicasts it into both shared memories (L2 weight traffic halves); a stage is refilled when the MMAs of
// BOTH CTAs have read it (tcgen05.commit multicast to both CTAs' "empty" barriers).
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void bulk_g2s_multicast(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint16_t mask) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "h"(mask) : "memory");
}
__device__ __forceinline__ void umma_commit_multicast(uint32_t bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(mask) : "memory");
}

// ---- cta_group::2 for the residual convolutions (KC32 = 8, TAPS = 9, N = 256): the two CTAs of a pair issue ONE M = 256 MMA
// for their two tiles.  Each CTA keeps only ITS half of every weight stage (128 of the 256 B rows, 8 KB): the tensor cores of
// the pair read both halves, so a CTA fetches 4 KB of A + 4 KB of B per MMA from its shared memory instead of 4 + 8 KB (the
// operand fetch sustains ~85 B/clk here; N = 256 at cta_group::1 needs 96).  The leader (rank 0) issues the MMAs; the
// follower's MMA warp walks the same loop and forwards "my A group / my weight half has landed" to the leader's barriers.
#ifndef SPB_CHESS_CTA2
#define SPB_CHESS_CTA2 0
#endif
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t cta_rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(cta_rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) { asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory"); }
__device__ __forceinline__ void umma2_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n}"
               ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma2_commit_multicast(uint32_t bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(mask) : "memory");
}
__host__ __device__ constexpr uint32_t make_idesc2(int N) {      // cta_group::2: M = 256 over the pair
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
}
__host__ __device__ constexpr bool conv_cta2(int kc32, int taps, int n) { return SPB_CHESS_CTA2 && kc32 == 8 && taps == 9 && n == 256; }

struct ConvArgs {
  const uint8_t* in;        // planar bf16 [KC32*4][plane_rows][8]
  uint8_t* out;             // planar bf16 [N/8][plane_rows][8] (EPI 0 / 1; EPI 1 adds the skip it reads from `out` itself)
  const uint8_t* w;         // weight stages, [kc32][tap][4 chunks][N][8] bf16
  const float* bias;        // [N]
  const uint32_t* count;    // positions in this batch (device)
  uint32_t plane_rows;
  float* logits;            // EPI 2: [slot][4672]
  const uint32_t* list;     // EPI 2: slot of position i (nullptr: identity)
  const float* vw;          // EPI 3: the value head's 1x1 conv weights [256] (model/chess.rs:61)
  float* vcell;             // EPI 3: [position of the batch][64] f32: that conv's output before bias and ReLU
};

// EPI_SKIP_RELU_VALUE: the torso's last conv; its epilogue also forms the value head's 1x1 conv (256 -> 1) of the cell it
// holds in registers, so the value head never reads the torso output back from HBM
enum { EPI_RELU = 0, EPI_SKIP_RELU = 1, EPI_LOGITS = 2, EPI_SKIP_RELU_VALUE = 3 };

template <int KC32, int TAPS, int N, int EPI>
struct ConvCfg {
  static constexpr int A_CHUNKS = KC32 * 4;
  static constexpr uint32_t A_BYTES = (uint32_t)A_CHUNKS * QA * 16;
  static constexpr bool CTA2 = conv_cta2(KC32, TAPS, N);
  static constexpr uint32_t STAGE_BYTES = 4u * N * 16;             // one weight stage in global memory
  static constexpr uint32_t SLOT_BYTES_B = CTA2 ? STAGE_BYTES / 2 : STAGE_BYTES;   // what a CTA keeps of it
  static constexpr int NST = CTA2 ? 2 * NSTAGE : NSTAGE;          // ring depth: the same 128 KB either way
  static constexpr uint32_t GROUP_BYTES = 4u * QA * 16;       // one 32-channel group of the A tile
  static constexpr uint32_t OFF_B = A_BYTES;
  static constexpr uint32_t OFF_BIAS = OFF_B + NST * SLOT_BYTES_B;
  static constexpr uint32_t OFF_VW = OFF_BIAS + 256 * 4;
  static constexpr uint32_t OFF_BAR = OFF_VW + (EPI == 3 ? 256 * 4 : 0);
  static constexpr uint32_t N_BARS = 28 + 3 * NST;             // a_full/empty[8], acc_full/empty[2], b_full/empty[NSTAGE], peer_a_full[8], peer_b_full[NSTAGE]
  static constexpr uint32_t SMEM = OFF_BAR + (N_BARS + 2) * 8;
};

template <int KC32, int TAPS, int N, int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(CONV_THREADS, 1) k_conv(const ConvArgs a) {
  using Cfg = ConvCfg<KC32, TAPS, N, EPI>;
  constexpr int NST = Cfg::NST;
  extern __shared__ __align__(1024) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar0 = sbase + Cfg::OFF_BAR;
  // barriers: a_full[8] a_empty[8] acc_full[2] acc_empty[2] b_full[NST] b_empty[NST], then the TMEM base word
  const uint32_t A_FULL = bar0, A_EMPTY = bar0 + 64, ACC_FULL = bar0 + 128, ACC_EMPTY = bar0 + 144, B_FULL = bar0 + 160,
                 B_EMPTY = bar0 + 160 + NST * 8;
  // cta_group::2, in the leader: the follower's A groups / weight halves have landed
  const uint32_t PEER_A_FULL = bar0 + 160 + 2 * NST * 8, PEER_B_FULL = PEER_A_FULL + 64;
  constexpr bool CTA2 = Cfg::CTA2;
  uint32_t* tmem_word = reinterpret_cast<uint32_t*>(smem + Cfg::OFF_BAR + Cfg::N_BARS * 8);
  float* s_bias = reinterpret_cast<float*>(smem + Cfg::OFF_BIAS);
  float* s_vw = reinterpret_cast<float*>(smem + Cfg::OFF_VW);

  const uint32_t boards = *a.count;
  const uint32_t n_tiles = tiles_for(boards);
  // pair p of the grid's CTA pairs takes tiles 2p and 2p+1 (an odd tail leaves one CTA a dummy tile beyond the batch: its
  // rows are allocated, its epilogue writes nothing), so both CTAs of a pair always run the same number of weight stages
  const uint32_t rank = cluster_ctarank();
  const uint32_t pair0 = blockIdx.x >> 1, n_pairs_grid = gridDim.x >> 1, n_pair_tiles = (n_tiles + 1u) >> 1;
  if (threadIdx.x == 0) {
    for (int i = 0; i < 8; ++i) { mbar_init(A_FULL + i * 8, 1); mbar_init(A_EMPTY + i * 8, 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(ACC_FULL + i * 8, 1); mbar_init(ACC_EMPTY + i * 8, CTA2 ? 8 : 4); }   // cta2: both CTAs' epilogue warps
    for (int i = 0; i < NST; ++i) { mbar_init(B_FULL + i * 8, 1); mbar_init(B_EMPTY + i * 8, CTA2 ? 1 : 2); }   // empty: both CTAs' MMAs / one pair commit
    if (CTA2) {
      for (int i = 0; i < 8; ++i) mbar_init(PEER_A_FULL + i * 8, 1);
      for (int i = 0; i < NST; ++i) mbar_init(PEER_B_FULL + i * 8, 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = threadIdx.x; i < N; i += CONV_THREADS) s_bias[i] = a.bias[i];
  if (EPI == EPI_SKIP_RELU_VALUE)
    for (int i = threadIdx.x; i < N; i += CONV_THREADS) s_vw[i] = a.vw[i];
  if (warp == 1) { if (CTA2) tmem_alloc2(smem_u32(tmem_word), 512); else tmem_alloc(smem_u32(tmem_word), 512); }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                                // the peer's barriers exist before anything is sent to them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_word;

  if (warp == 0) {
    // ---- producer ---------------------------------------------------------------------------------------------
    if (elect_one()) {
      uint32_t it = 0, st = 0;
      constexpr uint32_t HALF = Cfg::STAGE_BYTES / 2;
      for (uint32_t pt = pair0; pt < n_pair_tiles; pt += n_pairs_grid, ++it) {
        const uint32_t tile = 2u * pt + rank;
        const uint8_t* src = a.in + (size_t)tile * TILE_SPAN * 16;  // rows [LEAD + 144 tile - 16, + QA) of every plane
#pragma unroll 1
        for (int kc = 0; kc < KC32; ++kc) {
          // channel group kc of this tile's A: free once the 9 taps of the same group of the previous tile have been read
          mbar_wait_sleep(A_EMPTY + kc * 8, (it & 1u) ^ 1u);
          mbar_expect_tx(A_FULL + kc * 8, Cfg::GROUP_BYTES);
#pragma unroll
          for (int c = 0; c < 4; ++c)
            bulk_g2s(sbase + (uint32_t)(kc * 4 + c) * QA * 16, src + (size_t)(kc * 4 + c) * a.plane_rows * 16, QA * 16, A_FULL + kc * 8);
#pragma unroll 1
          for (int tap = 0; tap < TAPS; ++tap, ++st) {
            const uint32_t slot = st % NST;
            // both CTAs have read the slot's previous stage (cta_group::2: slots are released four at a time)
            if (!CTA2) mbar_wait_sleep(B_EMPTY + slot * 8, ((st / NST) & 1u) ^ 1u);
            else if ((st & 3u) == 0u) mbar_wait_sleep(B_EMPTY + (slot >> 2) * 8, ((st / NST) & 1u) ^ 1u);
            if (CTA2) {                                                          // this CTA's 128 B rows of the stage (packed contiguously)
              mbar_expect_tx(B_FULL + slot * 8, HALF);
              bulk_g2s(sbase + Cfg::OFF_B + slot * HALF, a.w + (size_t)(kc * TAPS + tap) * Cfg::STAGE_BYTES + rank * HALF, HALF, B_FULL + slot * 8);
            } else {
              mbar_expect_tx(B_FULL + slot * 8, Cfg::STAGE_BYTES);               // own half + the peer's half
              bulk_g2s_multicast(sbase + Cfg::OFF_B + slot * Cfg::STAGE_BYTES + rank * HALF,
                                 a.w + (size_t)(kc * TAPS + tap) * Cfg::STAGE_BYTES + rank * HALF, HALF, B_FULL + slot * 8, (uint16_t)3);
            }
          }
        }
      }
      // the peer's last "slot is free" signals must have landed in THIS CTA's barriers before it exits
      for (uint32_t k = 0; k < (uint32_t)NST && k < st; k += CTA2 ? 4u : 1u) {
        const uint32_t s2 = st - 1u - k;
        mbar_wait_sleep(B_EMPTY + (CTA2 ? (s2 % NST) >> 2 : s2 % NST) * 8, (s2 / NST) & 1u);
      }
    }
  } else if (warp == 1) {
    // ---- MMA issuer -------------------------------------------------------------------------------------------
    const bool issuer = elect_one();
    constexpr uint32_t DESC_HI_A = 9u | (1u << 14);                 // A: SBO = 9 rows = 144 B between core matrices, descriptor version 1
    constexpr uint32_t DESC_HI_B = (128u >> 4) | (1u << 14);        // B: SBO = 128 B
    constexpr uint32_t IDESC = CTA2 ? make_idesc2(N) : make_idesc(N);
    constexpr uint32_t NB = CTA2 ? N / 2 : N;                        // B rows in this CTA's shared memory
    // descriptor start addresses are CTA-relative 18-bit offsets: in a cluster the shared-window address of rank 1 carries
    // the CTA rank in its upper bits, which must not spill into the LBO field
    const uint32_t soff = sbase & 0x3FFFFu;
    const uint32_t a_lo_base = ((soff >> 4) + 16u) | ((uint32_t)QA << 16);   // row 16 of the buffer, LBO = QA rows
    const bool leader = !CTA2 || rank == 0;
    uint32_t it = 0, st = 0;
    for (uint32_t pt = pair0; pt < n_pair_tiles; pt += n_pairs_grid, ++it) {
      const uint32_t buf = it & 1u, par = (it >> 1) & 1u;
      if (leader) {
        mbar_wait(ACC_EMPTY + buf * 8, par ^ 1u);
        tc_fence_after();
      }
      const uint32_t d_tmem = tmem_base + buf * 256;
#pragma unroll 1
      for (int kc = 0; kc < KC32; ++kc) {
        mbar_wait(A_FULL + kc * 8, it & 1u);
        if (CTA2 && leader) mbar_wait(PEER_A_FULL + kc * 8, it & 1u);
        if (CTA2 && !leader && issuer) mbar_arrive_cluster(mapa_shared(PEER_A_FULL + kc * 8, 0));   // my A group has landed
        tc_fence_after();
#pragma unroll 1
        for (int tap = 0; tap < TAPS; ++tap, ++st) {
          const int shift = TAPS == 9 ? (tap / 3 - 1) * 9 + (tap % 3 - 1) : 0;
          const uint32_t slot = st % NST;
          mbar_wait(B_FULL + slot * 8, (st / NST) & 1u);
          // the follower forwards its weight halves four stages at a time (a remote arrival per stage would bound the loop)
          if (CTA2 && leader && (st & 3u) == 0u) mbar_wait(PEER_B_FULL + (slot >> 2) * 8, (st / NST) & 1u);
          if (CTA2 && !leader && issuer && (st & 3u) == 3u) mbar_arrive_cluster(mapa_shared(PEER_B_FULL + (slot >> 2) * 8, 0));
          tc_fence_after();
          if (issuer && leader) {
            const uint32_t b_lo_base = ((soff + Cfg::OFF_B + slot * Cfg::SLOT_BYTES_B) >> 4) | ((uint32_t)NB << 16);
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
              const uint32_t a_lo = a_lo_base + (uint32_t)(shift + (kc * 4 + kk * 2) * QA);
              const uint32_t b_lo = b_lo_base + (uint32_t)(kk * 2 * NB);
              if (CTA2) umma2_f16(d_tmem, ((uint64_t)DESC_HI_A << 32) | a_lo, ((uint64_t)DESC_HI_B << 32) | b_lo, IDESC, (tap | kc | kk) != 0);
              else umma_f16(d_tmem, ((uint64_t)DESC_HI_A << 32) | a_lo, ((uint64_t)DESC_HI_B << 32) | b_lo, IDESC, (tap | kc | kk) != 0);
            }
            if (!CTA2) umma_commit_multicast(B_EMPTY + slot * 8, (uint16_t)3);   // frees the slot in both CTAs
            else if ((st & 3u) == 3u) umma2_commit_multicast(B_EMPTY + (slot >> 2) * 8, (uint16_t)3);   // ... four slots
          }
          __syncwarp();
        }
        if (issuer && leader) {                                       // this channel group of the A tile has been read
          if (CTA2) umma2_commit_multicast(A_EMPTY + kc * 8, (uint16_t)3); else umma_commit(A_EMPTY + kc * 8);
        }
        __syncwarp();
      }
      if (issuer && leader) { if (CTA2) umma2_commit_multicast(ACC_FULL + buf * 8, (uint16_t)3); else umma_commit(ACC_FULL + buf * 8); }
      __syncwarp();
    }
  } else {
    // ---- epilogue ---------------------------------------------------------------------------------------------
    const int q = warp & 3;                                            // TMEM lane quadrant this warp may read
    uint32_t it = 0;
    for (uint32_t pt = pair0; pt < n_pair_tiles; pt += n_pairs_grid, ++it) {
      const uint32_t tile = 2u * pt + rank;
      const uint32_t buf = it & 1u, par = (it >> 1) & 1u;
      mbar_wait(ACC_FULL + buf * 8, par);
      tc_fence_after();
      // TMEM lane r = board row (r >> 3) of the tile, cell (r & 7)
      const uint32_t brow = tile * TILE_BROWS + (uint32_t)((q * 32 + lane) >> 3), x = (uint32_t)(lane & 7);
      const uint32_t board = brow / 9u, y = brow % 9u;
      const bool pad = y == 8u || board >= boards;                    // the shared zero row / beyond the batch: never written
      const uint32_t r_layout = brow * 9u + x;
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + buf * 256;
      if (EPI == EPI_LOGITS) {
        const uint32_t slot = (!pad && a.list) ? a.list[board] : board;
        float* dst = a.logits + (size_t)slot * SPB_CHESS_POLICY_SIZE + y * 8 + x;
#pragma unroll 1
        for (int c16 = 0; c16 < N / 16; ++c16) {
          uint32_t r[16];
          tmem_ld16(taddr + c16 * 16, r);
          tmem_ld_wait();
          if (!pad) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const int ch = c16 * 16 + j;
              if (ch < NET_MOVE_PLANES) dst[ch * 64] = __uint_as_float(r[j]) + s_bias[ch];
            }
          }
        }
      } else {
        uint8_t* orow = a.out + ((size_t)LEAD + r_layout) * 16;
        float vdot = 0.0f;
#pragma unroll 1
        for (int c32 = 0; c32 < N / 32; ++c32) {
          uint32_t r[32];
          tmem_ld16(taddr + c32 * 32, r);
          tmem_ld16(taddr + c32 * 32 + 16, r + 16);
          uint4 sk[4];
          if ((EPI == EPI_SKIP_RELU || EPI == EPI_SKIP_RELU_VALUE) && !pad) {
#pragma unroll
            for (int c = 0; c < 4; ++c) sk[c] = *reinterpret_cast<const uint4*>(orow + (size_t)(c32 * 4 + c) * a.plane_rows * 16);
          }
          tmem_ld_wait();
          if (!pad) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const int ch0 = c32 * 32 + c * 8;
              float v[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(r[c * 8 + j]) + s_bias[ch0 + j];
              if (EPI == EPI_SKIP_RELU || EPI == EPI_SKIP_RELU_VALUE) {
                const uint32_t s4[4] = {sk[c].x, sk[c].y, sk[c].z, sk[c].w};
#pragma unroll
                for (int j = 0; j < 4; ++j) { v[2 * j] += bf_lo(s4[j]); v[2 * j + 1] += bf_hi(s4[j]); }
              }
              if (EPI == EPI_SKIP_RELU_VALUE) {
#pragma unroll
                for (int j = 0; j < 8; ++j) vdot = fmaf(fmaxf(v[j], 0.f), s_vw[ch0 + j], vdot);
              }
              uint4 o;
              o.x = pack_bf16x2(fmaxf(v[0], 0.f), fmaxf(v[1], 0.f));
              o.y = pack_bf16x2(fmaxf(v[2], 0.f), fmaxf(v[3], 0.f));
              o.z = pack_bf16x2(fmaxf(v[4], 0.f), fmaxf(v[5], 0.f));
              o.w = pack_bf16x2(fmaxf(v[6], 0.f), fmaxf(v[7], 0.f));
              *reinterpret_cast<uint4*>(orow + (size_t)(c32 * 4 + c) * a.plane_rows * 16) = o;
            }
          }
        }
        if (EPI == EPI_SKIP_RELU_VALUE && !pad) a.vcell[(size_t)board * 64 + y * 8 + x] = vdot;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {                                                // cta_group::2: the leader's barrier collects both CTAs' epilogue warps
        if (CTA2 && rank != 0) mbar_arrive_cluster(mapa_shared(ACC_EMPTY + buf * 8, 0)); else mbar_arrive(ACC_EMPTY + buf * 8);
      }
    }
  }
  tc_fence_before();
  __syncwarp();
  __syncthreads();
  cluster_sync_all();                                                // no CTA leaves while its peer may still signal its barriers
  if (warp == 1) { if (CTA2) tmem_dealloc2(tmem_base, 512); else tmem_dealloc(tmem_base, 512); }
}

// ---- input planes (get_encoding, chess.rs:176-249) as the stem's A operand: [4 chunks][rows][8] bf16 ------------------
__global__ void k_encode_input(const Pos* pos, const uint32_t* reps, const uint32_t* list, const uint32_t* count, uint8_t* out, uint32_t plane_rows) {
  const uint32_t boards = *count;
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;          // row of the batch
  const uint32_t n_rows = tiles_for(boards) * TILE_SPAN;
  if (r >= n_rows) return;
  const uint32_t board = r / BOARD_ROWS, cell = r % BOARD_ROWS, row = cell / 9, col = cell % 9;
  float v[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = 0.0f;
  if (board < boards && row < 8 && col < 8) {
    const uint32_t slot = list ? list[board] : board;
    const Pos p = pos[slot];
    const uint32_t rp = reps[slot];
#pragma unroll
    for (int pl = 0; pl < NET_IN; ++pl) v[pl] = encode_plane(p, rp, pl, (int)row, (int)col);
  }
#pragma unroll
  for (int c = 0; c < IN_CHUNKS; ++c) {
    uint4 o;
    o.x = pack_bf16x2(v[c * 8 + 0], v[c * 8 + 1]);
    o.y = pack_bf16x2(v[c * 8 + 2], v[c * 8 + 3]);
    o.z = pack_bf16x2(v[c * 8 + 4], v[c * 8 + 5]);
    o.w = pack_bf16x2(v[c * 8 + 6], v[c * 8 + 7]);
    *reinterpret_cast<uint4*>(out + ((size_t)c * plane_rows + LEAD + r) * 16) = o;
  }
}

// ---- value head (model/chess.rs:61-70): 1x1 conv 256 -> 1 (formed in the last torso conv's epilogue: vcell), + bias, ReLU,
// Linear 64 -> 256, ReLU, Linear 256 -> 1, tanh.  One block of 256 threads per VH_POS positions: thread t owns hidden unit t
// and reads its 64 fc1 weights once for all of them.
constexpr int VH_POS = 8;
__global__ void __launch_bounds__(256) k_value_head(const float* vcell, const uint32_t* list, const uint32_t* count, const float* vconv_b,
                                                    const float* fc1_w, const float* fc1_b, const float* fc2_w, const float* fc2_b, float* values) {
  __shared__ float s_cell[VH_POS][64];
  __shared__ float s_red[VH_POS][8];
  const uint32_t n = *count, b0 = blockIdx.x * VH_POS;
  if (b0 >= n) return;
  const int t = threadIdx.x;
  const float vb = vconv_b[0];
  for (int i = t; i < VH_POS * 64; i += 256) {
    const uint32_t board = b0 + (uint32_t)(i >> 6);
    s_cell[i >> 6][i & 63] = board < n ? fmaxf(vcell[(size_t)board * 64 + (i & 63)] + vb, 0.0f) : 0.0f;
  }
  __syncthreads();
  float h[VH_POS];
  const float hb = fc1_b[t];
#pragma unroll
  for (int p = 0; p < VH_POS; ++p) h[p] = hb;
  for (int k = 0; k < 64; ++k) {
    const float w = fc1_w[k * 256 + t];                              // fc1_w is stored transposed [64][256]: coalesced over t
#pragma unroll
    for (int p = 0; p < VH_POS; ++p) h[p] += w * s_cell[p][k];
  }
  const float w2 = fc2_w[t];
#pragma unroll
  for (int p = 0; p < VH_POS; ++p) {
    float y = fmaxf(h[p], 0.0f) * w2;
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) y += __shfl_xor_sync(0xffffffffu, y, o);
    if ((t & 31) == 0) s_red[p][t >> 5] = y;
  }
  __syncthreads();
  if (t < VH_POS && b0 + (uint32_t)t < n) {
    float sum = fc2_b[0];
    for (int i = 0; i < 8; ++i) sum += s_red[t][i];
    const uint32_t board = b0 + (uint32_t)t;
    values[list ? list[board] : board] = tanhf(sum);
  }
}

// ---- host ------------------------------------------------------------------------------------------------------------
// Activation buffers of one evaluator batch.  Set 0 holds up to the engine's num_games positions (spb_chess_predict, the
// first half of the trees in the search), set 1 the second half of the trees (chess_engine.cu: two half-loops on two streams).
struct ActSet {
  uint32_t max_positions = 0;
  size_t plane_rows = 0;
  uint8_t* d_in = nullptr;      // [4][plane_rows][8] bf16
  uint8_t* d_x = nullptr;       // [32][plane_rows][8]
  uint8_t* d_y = nullptr;
  float* d_vcell = nullptr;     // [max_positions][64] f32: the value head's 1x1 conv, from the last torso conv's epilogue
};
struct Net {
  ActSet act[2];
  uint8_t* d_w = nullptr;       // weight image
  size_t w_bytes = 0;
  size_t off_conv[NET_CONV3] = {}, off_p1 = 0, off_p2 = 0;
  float* d_f = nullptr;         // f32 parameters: biases + value head
  size_t off_bias[NET_CONV3] = {}, off_bp1 = 0, off_bp2 = 0, off_vw = 0, off_vb = 0, off_f1w = 0, off_f1b = 0, off_f2w = 0, off_f2b = 0;
  bool loaded = false;
  bool attrs_set = false;
};

// weight stages of one conv: [kc32][tap][4 chunks][N][8] bf16; input channels padded to kc32*32, outputs to N
// cta_group::2 convolutions: a stage is two halves [rank][4 chunks][N/2][8], rank r = output channels r N/2 .. (r+1) N/2 - 1
static void pack_conv(const HostNet::Conv& cv, int kc32, int N, uint16_t* dst) {
  const int taps = cv.k * cv.k;
  const bool halves = conv_cta2(kc32, taps, N);
  const int NH = halves ? N / 2 : N;
  for (int tap = 0; tap < taps; ++tap)
    for (int kc = 0; kc < kc32; ++kc) {
      uint16_t* st = dst + ((size_t)kc * taps + tap) * 4 * N * 8;
      for (int n = 0; n < N; ++n)
        for (int kl = 0; kl < 32; ++kl) {
          const int k = kc * 32 + kl;
          const float w = (n < cv.oc && k < cv.ic) ? cv.w[((size_t)n * cv.ic + k) * taps + tap] : 0.0f;
          st[(size_t)(n / NH) * 4 * NH * 8 + ((size_t)(kl / 8) * NH + (n % NH)) * 8 + (kl % 8)] = f2bf(w);
        }
    }
}

Net* net_create(uint32_t max_positions, std::string* err) {
  Net* net = new (std::nothrow) Net();
  if (!net) { *err = "out of host memory"; return nullptr; }
  net->act[0].max_positions = max_positions;
  net->act[1].max_positions = std::max(1u, max_positions / 2u);
  size_t w = 0;
  for (int i = 0; i < NET_CONV3; ++i) { net->off_conv[i] = w; w += (size_t)9 * (i == 0 ? 1 : 8) * 4 * 256 * 16; }
  net->off_p1 = w; w += (size_t)8 * 4 * 256 * 16;
  net->off_p2 = w; w += (size_t)8 * 4 * 80 * 16;
  net->w_bytes = w;
  size_t f = 0;
  for (int i = 0; i < NET_CONV3; ++i) { net->off_bias[i] = f; f += 256; }
  net->off_bp1 = f; f += 256;
  net->off_bp2 = f; f += 256;
  net->off_vw = f; f += 256;
  net->off_vb = f; f += 8;
  net->off_f1w = f; f += 256 * 64;
  net->off_f1b = f; f += 256;
  net->off_f2w = f; f += 256;
  net->off_f2b = f; f += 8;
  bool ok = cudaMalloc(&net->d_w, net->w_bytes) == cudaSuccess && cudaMalloc(&net->d_f, f * 4) == cudaSuccess;
  for (int k = 0; k < 2 && ok; ++k) {
    ActSet& a = net->act[k];
    a.plane_rows = plane_rows_for(a.max_positions);
    const size_t plane = a.plane_rows * 16;
    ok = cudaMalloc(&a.d_in, IN_CHUNKS * plane) == cudaSuccess && cudaMalloc(&a.d_x, 32 * plane) == cudaSuccess &&
         cudaMalloc(&a.d_y, 32 * plane) == cudaSuccess && cudaMalloc(&a.d_vcell, (size_t)a.max_positions * 64 * 4) == cudaSuccess;
    if (ok) {                                                         // lead / tail rows are never written by a kernel: zero once
      cudaMemset(a.d_in, 0, IN_CHUNKS * plane);
      cudaMemset(a.d_x, 0, 32 * plane);
      cudaMemset(a.d_y, 0, 32 * plane);
    }
  }
  if (!ok) {
    *err = "out of device memory for the chess network's activations";
    net_destroy(net);
    return nullptr;
  }
  return net;
}

void net_destroy(Net* net) {
  if (!net) return;
  for (ActSet& a : net->act) { cudaFree(a.d_in); cudaFree(a.d_x); cudaFree(a.d_y); cudaFree(a.d_vcell); }
  cudaFree(net->d_w); cudaFree(net->d_f);
  delete net;
}

bool net_loaded(const Net* net) { return net && net->loaded; }
void net_set_loaded(Net* net, bool ok) { net->loaded = ok; }

NetImage net_image(Net* net) {
  NetImage m;
  m.d_w = net->d_w; m.w_bytes = net->w_bytes;
  m.d_f = net->d_f; m.f_count = net->off_f2b + 8;
  for (int i = 0; i < NET_CONV3; ++i) { m.off_conv[i] = net->off_conv[i]; m.off_bias[i] = net->off_bias[i]; }
  m.off_p1 = net->off_p1; m.off_p2 = net->off_p2;
  m.off_bp1 = net->off_bp1; m.off_bp2 = net->off_bp2; m.off_vw = net->off_vw; m.off_vb = net->off_vb;
  m.off_f1w = net->off_f1w; m.off_f1b = net->off_f1b; m.off_f2w = net->off_f2w; m.off_f2b = net->off_f2b;
  m.res_halves = conv_cta2(8, 9, 256);
  return m;
}

double net_flops_per_position() {
  double f = 2.0 * 64 * NET_IN * 9 * 256;                               // stem
  f += 20.0 * 2.0 * 64 * 256 * 9 * 256;                                 // residual convs
  f += 2.0 * 64 * 256 * 256 + 2.0 * 64 * 256 * NET_MOVE_PLANES;         // policy head
  f += 2.0 * 64 * 256 + 2.0 * 64 * 256 + 2.0 * 256;                     // value head
  return f;
}

bool net_upload(Net* net, const HostNet& h, std::string* err) {
  std::vector<uint16_t> img(net->w_bytes / 2, 0);
  for (int i = 0; i < NET_CONV3; ++i) pack_conv(h.conv3[i], i == 0 ? 1 : 8, 256, img.data() + net->off_conv[i] / 2);
  pack_conv(h.p1, 8, 256, img.data() + net->off_p1 / 2);
  pack_conv(h.p2, 8, 80, img.data() + net->off_p2 / 2);
  std::vector<float> f(net->off_f2b + 8, 0.0f);
  for (int i = 0; i < NET_CONV3; ++i) std::copy(h.conv3[i].b.begin(), h.conv3[i].b.end(), f.begin() + net->off_bias[i]);
  std::copy(h.p1.b.begin(), h.p1.b.end(), f.begin() + net->off_bp1);
  std::copy(h.p2.b.begin(), h.p2.b.end(), f.begin() + net->off_bp2);
  std::copy(h.vconv.w.begin(), h.vconv.w.end(), f.begin() + net->off_vw);
  f[net->off_vb] = h.vconv.b[0];
  for (int o = 0; o < 256; ++o)
    for (int k = 0; k < 64; ++k) f[net->off_f1w + (size_t)k * 256 + o] = h.fc1_w[(size_t)o * 64 + k];   // transposed for the value-head kernel
  std::copy(h.fc1_b.begin(), h.fc1_b.end(), f.begin() + net->off_f1b);
  std::copy(h.fc2_w.begin(), h.fc2_w.end(), f.begin() + net->off_f2w);
  f[net->off_f2b] = h.fc2_b[0];
  if (cudaMemcpy(net->d_w, img.data(), net->w_bytes, cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemcpy(net->d_f, f.data(), f.size() * 4, cudaMemcpyHostToDevice) != cudaSuccess) {
    *err = std::string("weight upload: ") + cudaGetErrorString(cudaGetLastError());
    return false;
  }
  net->loaded = true;
  return true;
}

template <int KC32, int TAPS, int N, int EPI>
static cudaError_t launch_conv(const ActSet& act, const ConvArgs& a, cudaStream_t stream) {
  using Cfg = ConvCfg<KC32, TAPS, N, EPI>;
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(k_conv<KC32, TAPS, N, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
    if (e != cudaSuccess) return e;
    attr = true;
  }
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const uint32_t grid = 2u * std::min<uint32_t>((uint32_t)sms / 2u, (tiles_for(act.max_positions) + 1u) / 2u);   // CTA pairs
  k_conv<KC32, TAPS, N, EPI><<<grid, CONV_THREADS, Cfg::SMEM, stream>>>(a);
  return cudaGetLastError();
}

cudaError_t net_forward(Net* net, int set, const Pos* pos, const uint32_t* reps, const uint32_t* list, const uint32_t* count_dev, float* logits,
                        float* values, cudaStream_t stream, uint32_t* launched) {
  const ActSet& act = net->act[set];
  const uint32_t plane_rows = (uint32_t)act.plane_rows;
  const uint32_t max_rows = tiles_for(act.max_positions) * TILE_SPAN;
  uint32_t n = 0;
  cudaError_t e;
  k_encode_input<<<(max_rows + 127) / 128, 128, 0, stream>>>(pos, reps, list, count_dev, act.d_in, plane_rows);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  ++n;
  ConvArgs a{};
  a.count = count_dev; a.plane_rows = plane_rows; a.list = list; a.logits = logits;
  // stem: x = relu(bn(conv(in)))
  a.in = act.d_in; a.out = act.d_x; a.w = net->d_w + net->off_conv[0]; a.bias = net->d_f + net->off_bias[0];
  if ((e = launch_conv<1, 9, 256, EPI_RELU>(act, a, stream)) != cudaSuccess) return e;
  ++n;
  for (int b = 0; b < NET_BLOCKS; ++b) {                               // resnet_block, model/mod.rs:152-166
    a.in = act.d_x; a.out = act.d_y; a.w = net->d_w + net->off_conv[1 + 2 * b]; a.bias = net->d_f + net->off_bias[1 + 2 * b];
    if ((e = launch_conv<8, 9, 256, EPI_RELU>(act, a, stream)) != cudaSuccess) return e;
    a.in = act.d_y; a.out = act.d_x; a.w = net->d_w + net->off_conv[2 + 2 * b]; a.bias = net->d_f + net->off_bias[2 + 2 * b];
    // x = relu(x + f(x)), in place; the last block's epilogue also forms the value head's 1x1 conv
    if (b + 1 < NET_BLOCKS) e = launch_conv<8, 9, 256, EPI_SKIP_RELU>(act, a, stream);
    else { a.vw = net->d_f + net->off_vw; a.vcell = act.d_vcell; e = launch_conv<8, 9, 256, EPI_SKIP_RELU_VALUE>(act, a, stream); }
    if (e != cudaSuccess) return e;
    n += 2;
  }
  // policy head: y = relu(conv1x1(x)); logits = conv1x1(y)
  a.in = act.d_x; a.out = act.d_y; a.w = net->d_w + net->off_p1; a.bias = net->d_f + net->off_bp1;
  if ((e = launch_conv<8, 1, 256, EPI_RELU>(act, a, stream)) != cudaSuccess) return e;
  a.in = act.d_y; a.out = nullptr; a.w = net->d_w + net->off_p2; a.bias = net->d_f + net->off_bp2;
  if ((e = launch_conv<8, 1, 80, EPI_LOGITS>(act, a, stream)) != cudaSuccess) return e;
  n += 2;
  k_value_head<<<(act.max_positions + VH_POS - 1) / VH_POS, 256, 0, stream>>>(act.d_vcell, list, count_dev, net->d_f + net->off_vb, net->d_f + net->off_f1w,
                                                                              net->d_f + net->off_f1b, net->d_f + net->off_f2w, net->d_f + net->off_f2b, values);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  ++n;
  if (launched) *launched = n;
  return cudaSuccess;
}

// Re-runs one residual convolution (k_conv<8, 9, 256, EPI_RELU>: x -> y, layer 1; y is scratch between blocks) on the
// activations the last forward left in HBM, `iters` launches between two CUDA events on `stream`.
cudaError_t net_time_conv(Net* net, const uint32_t* count_dev, uint32_t iters, cudaStream_t stream, cudaEvent_t ev0, cudaEvent_t ev1, float* avg_ms) {
  const ActSet& act = net->act[0];
  ConvArgs a{};
  a.count = count_dev; a.plane_rows = (uint32_t)act.plane_rows;
  a.in = act.d_x; a.out = act.d_y; a.w = net->d_w + net->off_conv[1]; a.bias = net->d_f + net->off_bias[1];
  cudaError_t e;
  if ((e = launch_conv<8, 9, 256, EPI_RELU>(act, a, stream)) != cudaSuccess) return e;   // warm
  if ((e = cudaEventRecord(ev0, stream)) != cudaSuccess) return e;
  for (uint32_t i = 0; i < iters; ++i)
    if ((e = launch_conv<8, 9, 256, EPI_RELU>(act, a, stream)) != cudaSuccess) return e;
  if ((e = cudaEventRecord(ev1, stream)) != cudaSuccess) return e;
  if ((e = cudaEventSynchronize(ev1)) != cudaSuccess) return e;
  float ms = 0.f;
  if ((e = cudaEventElapsedTime(&ms, ev0, ev1)) != cudaSuccess) return e;
  *avg_ms = ms / (float)iters;
  return cudaSuccess;
}

int32_t net_forward_leaves(spb_chess_engine* e, int set, const uint32_t* list, const uint32_t* count_dev, cudaStream_t stream, uint32_t* launched) {
  SPB_CUDA(e, net_forward(e->net, set, e->T.leaf_pos, e->T.leaf_reps, list, count_dev, e->T.eval_logits, e->T.eval_value, stream, launched));
  return SPB_OK;
}

// ---- spb_chess_predict: Model::predict (model/mod.rs:36-98) for explicit states -----------------------------------------
// legal moves, repetition count and status of every state (one warp each), for the encoding's plane 16 and the mask
__global__ void __launch_bounds__(128) k_predict_prepare(const Pos* states, const unsigned long long* history, uint32_t n, Move* moves,
                                                         uint32_t* nmoves, uint32_t* reps, uint32_t* error) {
  __shared__ WarpScratch s_ws[4];
  const int lane = threadIdx.x & 31;
  WarpScratch& ws = s_ws[threadIdx.x >> 5];
  const uint32_t i = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (i >= n) return;
  const Pos p = states[i];
  const int m = warp_legal_moves(p, lane, ws, error);
  const unsigned long long h = warp_list_hash(ws, m, lane);
  const uint32_t hl = history ? min(p.hist_len, (uint32_t)SPB_CHESS_MAX_HISTORY) : 0u;
  const uint32_t r = warp_repetitions(h, history + (size_t)i * SPB_CHESS_MAX_HISTORY, hl, ws, 0, lane);
  for (int k = lane; k < m; k += 32) moves[(size_t)i * MAX_MOVES + k] = ws.moves[k];
  if (lane == 0) { nmoves[i] = (uint32_t)m; reps[i] = r; }
}

// softmax over the 4,672 logits (model/mod.rs:64), then mask_invalid_actions (chess.rs:251-271): legal cells / their sum
__global__ void __launch_bounds__(256) k_predict_mask(const float* logits, const Pos* states, const Move* moves, const uint32_t* nmoves, uint32_t n,
                                                      float* policies) {
  __shared__ float s_red[8];
  __shared__ float s_bcast;
  const uint32_t i = blockIdx.x;
  if (i >= n) return;
  const float* l = logits + (size_t)i * SPB_CHESS_POLICY_SIZE;
  float* out = policies + (size_t)i * SPB_CHESS_POLICY_SIZE;
  const int t = threadIdx.x;
  auto block_reduce = [&](float v, bool is_max) {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) { const float u = __shfl_xor_sync(0xffffffffu, v, o); v = is_max ? fmaxf(v, u) : v + u; }
    if ((t & 31) == 0) s_red[t >> 5] = v;
    __syncthreads();
    if (t == 0) { float r = s_red[0]; for (int k = 1; k < 8; ++k) r = is_max ? fmaxf(r, s_red[k]) : r + s_red[k]; s_bcast = r; }
    __syncthreads();
    const float r = s_bcast;
    __syncthreads();
    return r;
  };
  float mx = -INFINITY;
  for (int k = t; k < SPB_CHESS_POLICY_SIZE; k += 256) mx = fmaxf(mx, l[k]);
  mx = block_reduce(mx, true);
  float z = 0.0f;
  for (int k = t; k < SPB_CHESS_POLICY_SIZE; k += 256) { z += __expf(l[k] - mx); out[k] = 0.0f; }
  z = block_reduce(z, false);
  __syncthreads();
  const int side = states[i].side;
  const uint32_t m = nmoves[i];
  float s = 0.0f;
  for (uint32_t k = t; k < m; k += 256) s += __expf(l[policy_index(side, moves[(size_t)i * MAX_MOVES + k])] - mx) / z;
  s = block_reduce(s, false);
  for (uint32_t k = t; k < m; k += 256) {
    const int idx = policy_index(side, moves[(size_t)i * MAX_MOVES + k]);
    out[idx] = (__expf(l[idx] - mx) / z) / s;
  }
}

}  // namespace chess
}  // namespace spb

namespace ch = spb::chess;

extern "C" {

int32_t spb_chess_load_weights(spb_chess_engine* e, const void* blob, size_t n) {
  SPB_GUARD(e);
  SPB_ARG(e, blob && n > 8, "null / empty weight blob");
  ch::HostNet host;
  std::string err;
  if (!ch::parse_safetensors_chess(blob, n, &host, &err)) { e->set_error("spb_chess_load_weights: " + err); return SPB_ERR_WEIGHTS; }
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  if (!e->net) {
    e->net = ch::net_create(e->T.G, &err);
    if (!e->net) { e->set_error("spb_chess_load_weights: " + err); return SPB_ERR_NOMEM; }
  }
  if (!ch::net_upload(e->net, host, &err)) { e->set_error("spb_chess_load_weights: " + err); return SPB_ERR_CUDA; }
  return SPB_OK;
}

int32_t spb_chess_check_weights(const void* blob, size_t n, char* err, size_t err_cap) {
  if (err && err_cap) err[0] = 0;
  if (!blob) return SPB_ERR_ARG;
  ch::HostNet host;
  std::string msg;
  if (!ch::parse_safetensors_chess(blob, n, &host, &msg)) {
    if (err && err_cap) { std::strncpy(err, msg.c_str(), err_cap - 1); err[err_cap - 1] = 0; }
    return SPB_ERR_WEIGHTS;
  }
  return SPB_OK;
}

int32_t spb_chess_time_conv(spb_chess_engine* e, uint32_t iters, float* avg_ms, uint32_t* n_positions, double* flops_per_launch,
                            double* flops_per_position) {
  SPB_GUARD(e);
  SPB_ARG(e, avg_ms && n_positions && flops_per_launch && flops_per_position && iters > 0, "bad argument");
  SPB_ARG(e, e->net && ch::net_loaded(e->net), "no weights loaded (spb_chess_load_weights)");
  uint32_t n = 0;
  SPB_CUDA(e, cudaMemcpyAsync(&n, e->T.eval_count, 4, cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  SPB_ARG(e, n > 0, "no evaluator batch resident (run spb_chess_search first)");
  SPB_CUDA(e, ch::net_time_conv(e->net, e->T.eval_count, iters, e->stream, e->ev0, e->ev1, avg_ms));
  e->launches += iters + 1;
  *n_positions = n;
  *flops_per_launch = (double)n * 2.0 * 64 * 256 * 9 * 256;           // algorithmic: the 64 real cells of a position
  *flops_per_position = ch::net_flops_per_position();
  return SPB_OK;
}

int32_t spb_chess_predict(spb_chess_engine* e, const spb_chess_state* states, const uint64_t* history, uint32_t n, float* policies, float* values,
                          float* raw_logits) {
  SPB_GUARD(e);
  if (n == 0) return SPB_OK;
  SPB_ARG(e, states, "null states");
  SPB_ARG(e, e->net && ch::net_loaded(e->net), "no weights loaded (spb_chess_load_weights)");
  SPB_ARG(e, n <= e->T.G, "more states than the engine's num_games (the network's batch capacity)");
  const size_t hist_bytes = (size_t)n * SPB_CHESS_MAX_HISTORY * 8, row_bytes = (size_t)n * SPB_CHESS_POLICY_SIZE * 4;
  spb::StageLayout L;
  const size_t o_states = L.take((size_t)n * sizeof(ch::Pos)), o_hist = L.take(history ? hist_bytes : 0), o_moves = L.take((size_t)n * ch::MAX_MOVES * sizeof(ch::Move));
  const size_t o_nmoves = L.take((size_t)n * 4), o_reps = L.take((size_t)n * 4), o_count = L.take(4), o_logits = L.take(row_bytes), o_values = L.take((size_t)n * 4);
  const size_t o_pol = L.take(policies ? row_bytes : 0);
  if (int32_t rc = e->ensure_stage(L.bytes, 0)) return rc;
  auto* d_states = e->d_at<ch::Pos>(o_states);
  auto* d_hist = history ? e->d_at<unsigned long long>(o_hist) : nullptr;
  auto* d_moves = e->d_at<ch::Move>(o_moves);
  auto* d_nmoves = e->d_at<uint32_t>(o_nmoves);
  auto* d_reps = e->d_at<uint32_t>(o_reps);
  auto* d_count = e->d_at<uint32_t>(o_count);
  auto* d_logits = e->d_at<float>(o_logits);
  auto* d_values = e->d_at<float>(o_values);
  auto* d_pol = policies ? e->d_at<float>(o_pol) : nullptr;
  SPB_CUDA(e, cudaMemcpyAsync(d_states, states, (size_t)n * sizeof(ch::Pos), cudaMemcpyHostToDevice, e->stream));
  if (history) SPB_CUDA(e, cudaMemcpyAsync(d_hist, history, hist_bytes, cudaMemcpyHostToDevice, e->stream));
  SPB_CUDA(e, cudaMemcpyAsync(d_count, &n, 4, cudaMemcpyHostToDevice, e->stream));
  ch::k_predict_prepare<<<(n + 3) / 4, 128, 0, e->stream>>>(d_states, d_hist, n, d_moves, d_nmoves, d_reps, e->T.error);
  SPB_CUDA(e, cudaGetLastError());
  uint32_t launched = 0;
  SPB_CUDA(e, ch::net_forward(e->net, 0, d_states, d_reps, nullptr, d_count, d_logits, d_values, e->stream, &launched));
  e->launches += 1 + launched;
  if (policies) {
    ch::k_predict_mask<<<n, 256, 0, e->stream>>>(d_logits, d_states, d_moves, d_nmoves, n, d_pol);
    SPB_CUDA(e, cudaGetLastError());
    ++e->launches;
    SPB_CUDA(e, cudaMemcpyAsync(policies, d_pol, row_bytes, cudaMemcpyDeviceToHost, e->stream));
  }
  if (values) SPB_CUDA(e, cudaMemcpyAsync(values, d_values, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
  if (raw_logits) SPB_CUDA(e, cudaMemcpyAsync(raw_logits, d_logits, row_bytes, cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  return e->check_device_errors();
}

}  // extern "C"
