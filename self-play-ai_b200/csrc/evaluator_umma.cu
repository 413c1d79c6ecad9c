// evaluator_umma.cu — the fused policy/value network on tcgen05 tensor cores (sm_100a).
//
// Replaces Net::forward (ref: src/model/mod.rs:152-184, src/model/connect_four.rs:50-81, src/model/tictactoe.rs:50-81)
// and the tensor part of Model::predict (src/model/mod.rs:60-67,95).  One persistent CTA per SM runs the whole network
// on batches of <= NB boards with the activations resident in shared memory:
//   warp 0      weight producer: cp.async.bulk of the BN-folded bf16 weights into a 3-group ring (mbarrier complete_tx)
//   warp 1      MMA issuer: tcgen05.mma.cta_group::1.kind::f16, M = 128, accumulators in TMEM (two sets of 192 columns)
//   warp 2      stager: fetches the leaf positions of the next batch and writes their encoding (get_encoding,
//               connect_four.rs:242-259) as the stem's input
//   warp 3      publisher: results to global memory, evaluated trees to the ready ring
//   warps 4-11  epilogue: tcgen05.ld -> +bias (+skip) -> ReLU -> bf16 -> the other activation buffer; Linear heads,
//               softmax, tanh
//   warps 12-15 (asynchronous search pipeline only) tree warps: expand + backup + select of mcts.rs, see async.cuh
// Work comes either from a static list (spb_predict, lock-step pipeline: RING = false) or from the leaf ring of the
// asynchronous search pipeline (RING = true), where the kernel stays resident for a whole spb_search.
//
// A 3x3 conv is an implicit GEMM by row shift: a board is stored as 7 rows x 8 cells (one zero pad column, one zero pad
// row shared with the next board), so tap (dy,dx) is the constant row offset dy*8+dx of the UMMA descriptor's start
// address.  Measured on B200 (tools/umma_probe.cu T5): one thread issues one tcgen05.mma per ~46 cycles and an
// M=128,N=64,K=16 MMA needs 48 cycles of operand fetch, so one MMA per tap is bound by ISSUE + shared-memory fetch of A
// (4 KB per MMA, re-read for every tap), not by the tensor pipe (32 cycles).  Therefore the three taps of a kernel row
// (kx = 0, +1, -1) share ONE A fetch: their weights sit side by side as an N = 192 B operand, so one MMA (96 cycles,
// tensor-bound) yields D (columns 0..63, centre tap, final position), E (columns 64..127, right tap, computed one row
// early) and F (columns 128..191, left tap, one row late).  12 MMAs per tile-layer instead of 36; the epilogue forms
// out[r] = D[r] + E[r+1] + F[r-1] with two warp shuffles per channel — rows 32k-1 are pad cells, so lane 31 never needs
// E of the next warp and lane 0 takes F = 0 (F of a pad-column row is a sum over pad-column cells, which are zero).
// The fused head conv (N = 3 x 48) has the same form; the stem (one K step, 3 input planes) issues nine N = 64 MMAs, one per
// tap, into one accumulator: its epilogue needs no shuffles, and its phase is paced by the epilogue warps, not the tensor pipe.  Accumulators: two sets of 192 TMEM
// columns used in rotation by the CTA's tile sequence (batch, layer, tile); the spare 2 x 64 columns carry the skip
// connection of the residual blocks from the epilogue that produced it to the epilogue that adds it.
#include <cuda_bf16.h>

#include <cstring>
#include <mutex>

#include "bf16.cuh"
#include "evaluator_umma.cuh"
#include "umma_ptx.cuh"

namespace spb {
namespace umma {

// ---------------------------------------------------------------------------------------------------
// geometry
// ---------------------------------------------------------------------------------------------------
template <class G>
struct Geo {
  static constexpr int W8 = (G::COLS == 7) ? 8 : 4;          // padded row width
  static constexpr int RP = G::ROWS + 1;                     // rows incl. the shared zero pad row
  static constexpr int BS = W8 * RP;                         // rows per board (56 / 16)
  static constexpr int NT = 4;                               // tiles per batch
  static constexpr int NB = (NT * 128) / BS;                 // boards per batch (9 / 32)
  static constexpr int LEAD = 16;                            // zero rows in front (taps reach back W8+1)
  static constexpr int Q = LEAD + NT * 128 + 16;             // rows of an activation buffer
  static constexpr int P = G::ROWS * G::COLS;
  static constexpr int APAD = (G::A <= 8) ? 8 : 16;          // policy FC weights per (pos, channel), bf16
};

constexpr int N_LAYERS = 10;          // stem, 8 residual convs, fused head conv
constexpr int HEAD_N = 48;            // 32 policy + 3 value + 13 zero output channels
constexpr int SLOT_BYTES = 8192;      // one tap of a 64->64 layer
constexpr int N_SLOTS = 9;

__host__ __device__ constexpr int layer_n(int l) { return l == 9 ? HEAD_N : 64; }
__host__ __device__ constexpr int layer_kchunks(int l) { return l == 0 ? 2 : 8; }
__host__ __device__ constexpr int layer_tap_bytes(int l) { return layer_kchunks(l) * layer_n(l) * 16; }
__host__ __device__ constexpr size_t layer_offset(int l) {
  return l == 0 ? 0 : (size_t)9 * 2048 + (size_t)(l - 1) * 9 * SLOT_BYTES;
}
constexpr size_t OFF_BIAS = (size_t)9 * 2048 + (size_t)8 * 9 * SLOT_BYTES + (size_t)9 * 6144;   // 663,552
constexpr size_t OFF_WP = OFF_BIAS + (size_t)N_LAYERS * 64 * 4;
template <class G> __host__ __device__ constexpr size_t off_wv() { return OFF_WP + (size_t)G::A * Geo<G>::P * 32 * 4; }   // policy: f32 [A][P][32]
template <class G> __host__ __device__ constexpr size_t off_fcb() { return off_wv<G>() + (size_t)Geo<G>::P * 8 * 4; }        // value: f32 [P][8]
template <class G> __host__ __device__ constexpr size_t image_bytes() { return off_fcb<G>() + 32 * 4; }

// ---------------------------------------------------------------------------------------------------
// host: weight image
// ---------------------------------------------------------------------------------------------------
template <class G>
static ImageLayout image_layout_t() {
  ImageLayout L;
  for (int l = 0; l < N_LAYERS; ++l) {
    L.layer_offset[l] = layer_offset(l);
    L.layer_n[l] = layer_n(l);
    L.layer_kchunks[l] = layer_kchunks(l);
  }
  L.off_bias = OFF_BIAS; L.off_wp = OFF_WP; L.off_wv = off_wv<G>(); L.off_fcb = off_fcb<G>(); L.bytes = image_bytes<G>();
  return L;
}

ImageLayout image_layout(int game) { return game == SPB_GAME_CONNECT4 ? image_layout_t<Connect4>() : image_layout_t<TicTacToe>(); }

template <class G>
static void pack_t(const HostNet& net, std::vector<uint8_t>* out) {
  using Ge = Geo<G>;
  out->assign(image_bytes<G>(), 0);
  uint8_t* img = out->data();
  // Every conv layer but the stem in the kx-triple form: per kernel row ky one block [KC chunks][3N n][8] bf16 whose B rows are the
  // centre tap (n < N), the right tap (N <= n < 2N) and the left tap (2N <= n < 3N) of that kernel row — one MMA of
  // width 3N per K step serves all three taps from ONE fetch of A.  3 blocks per layer = the 3 ring groups.
  // The stem (K = 16: one K step) keeps one block [2 chunks][64 n][8] per tap, tap = ky*3 + kx: its 9 small MMAs cost the
  // tensor pipe nothing where it runs (behind the head conv of the previous batch, whose phase is paced by the epilogue
  // warps), and its epilogue needs no shuffles.
  for (int tap = 0; tap < 9; ++tap) {
    const HostNet::Conv& cv = net.conv[0];
    uint16_t* blk = reinterpret_cast<uint16_t*>(img + layer_offset(0) + (size_t)tap * layer_tap_bytes(0));
    for (int n = 0; n < 64; ++n)
      for (int k = 0; k < 16 && k < cv.ic; ++k)
        blk[((size_t)(k / 8) * 64 + n) * 8 + (k % 8)] = f2bf(cv.w[((size_t)n * cv.ic + k) * 9 + tap]);   // [OC][IC][ky][kx]
  }
  for (int l = 1; l < N_LAYERS; ++l) {
    const int N = layer_n(l), KC = layer_kchunks(l);
    const int n_real = l == 9 ? NET_POLICY_CH + NET_VALUE_CH : 64;
    for (int ky = 0; ky < 3; ++ky) {
      uint16_t* blk = reinterpret_cast<uint16_t*>(img + layer_offset(l) + (size_t)ky * 3 * layer_tap_bytes(l));
      for (int n = 0; n < n_real; ++n) {
        const HostNet::Conv& cv = l < 9 ? net.conv[l] : (n < NET_POLICY_CH ? net.conv[9] : net.conv[10]);
        const int oc = (l == 9 && n >= NET_POLICY_CH) ? n - NET_POLICY_CH : n;
        for (int k = 0; k < KC * 8 && k < cv.ic; ++k) {
          const float* w9 = &cv.w[((size_t)oc * cv.ic + k) * 9 + ky * 3];   // [OC][IC][ky][kx]: kx = 0 left, 1 centre, 2 right
          uint16_t* row = blk + ((size_t)(k / 8) * 3 * N) * 8 + (k % 8);
          row[(size_t)n * 8] = f2bf(w9[1]);
          row[(size_t)(N + n) * 8] = f2bf(w9[2]);
          row[(size_t)(2 * N + n) * 8] = f2bf(w9[0]);
        }
      }
    }
  }
  float* bias = reinterpret_cast<float*>(img + OFF_BIAS);
  for (int l = 0; l < 9; ++l)
    for (int n = 0; n < 64; ++n) bias[l * 64 + n] = net.conv[l].b[n];
  for (int n = 0; n < NET_POLICY_CH; ++n) bias[9 * 64 + n] = net.conv[9].b[n];
  for (int n = 0; n < NET_VALUE_CH; ++n) bias[9 * 64 + NET_POLICY_CH + n] = net.conv[10].b[n];
  // policy Linear: weight[a][ch*P + pos] -> f32 [a][pos][ch] (one 32-byte run per (output, position, 8-channel chunk))
  float* wp = reinterpret_cast<float*>(img + OFF_WP);
  for (int a = 0; a < G::A; ++a)
    for (int pos = 0; pos < Ge::P; ++pos)
      for (int ch = 0; ch < NET_POLICY_CH; ++ch)
        wp[((size_t)a * Ge::P + pos) * NET_POLICY_CH + ch] = net.pfc_w[(size_t)a * NET_POLICY_CH * Ge::P + (size_t)ch * Ge::P + pos];
  // value Linear: weight[0][ch*P + pos] -> f32 [pos][8] (channels 3..7 zero)
  float* wv = reinterpret_cast<float*>(img + off_wv<G>());
  for (int pos = 0; pos < Ge::P; ++pos)
    for (int ch = 0; ch < NET_VALUE_CH; ++ch) wv[pos * 8 + ch] = net.vfc_w[(size_t)ch * Ge::P + pos];
  float* fcb = reinterpret_cast<float*>(img + off_fcb<G>());
  for (int a = 0; a < G::A; ++a) fcb[a] = net.pfc_b[a];
  fcb[16] = net.vfc_b[0];
}

void pack_weights(const HostNet& net, std::vector<uint8_t>* out) {
  if (net.game == SPB_GAME_CONNECT4) pack_t<Connect4>(net, out);
  else pack_t<TicTacToe>(net, out);
}

// Issues the MMAs of one (layer, tile) in the kx-triple form: per kernel row ky, KSTEPS MMAs of width NP = 3N (centre |
// right | left taps) with A shifted by (ky-1)*W8 rows.  Ring group ky (3 slots = 24 KB) holds the row's block; K step kk
// reads the K chunks 2kk, 2kk+1 of A (stride Q rows) and of B (stride NP rows).  3 x KSTEPS MMAs per tile-layer (12 for a
// residual conv instead of 36 one-tap MMAs): A is fetched from shared memory once per kernel row and K step.
template <int W8, int Q, int KSTEPS, int NP>
__device__ __forceinline__ void issue_tile_triple(bool issuer, uint32_t a_lo_tile, uint32_t b_lo_base, uint32_t d_tmem,
                                                  bool first_tile, bool last_tile, uint32_t w_par, uint32_t bar_base,
                                                  uint32_t mid_bar, uint32_t mid_par) {
  constexpr uint32_t DESC_HI = (128u >> 4) | (1u << 14);          // SBO = 128 B, descriptor version 1
  constexpr uint32_t IDESC = make_idesc(NP);
#pragma unroll
  for (int ky = 0; ky < 3; ++ky) {
    const int shift = (ky - 1) * W8;
    if (ky == 2 && mid_bar) {                                     // the bottom kernel row reads the first rows of the next tile
      mbar_wait(mid_bar, mid_par);
      tc_fence_after();
    }
    if (first_tile) {                                             // w_full[ky]: the ring group of this kernel row
      mbar_wait(bar_base + (uint32_t)ky * 8u, w_par);
      tc_fence_after();
    }
    if (issuer) {
#pragma unroll
      for (int kk = 0; kk < KSTEPS; ++kk) {
        const uint32_t a_lo = a_lo_tile + (uint32_t)(shift + kk * 2 * Q);
        const uint32_t b_lo = (b_lo_base + (uint32_t)(3 * ky) * (SLOT_BYTES >> 4) + (uint32_t)(kk * 2 * NP)) | ((uint32_t)NP << 16);
        umma_f16(d_tmem, ((uint64_t)DESC_HI << 32) | a_lo, ((uint64_t)DESC_HI << 32) | b_lo, IDESC, (ky | kk) != 0);
      }
      if (last_tile) umma_commit(bar_base + (uint32_t)(N_SLOTS + ky) * 8u);                        // w_empty[ky]
    }
    __syncwarp();
  }
}

// The stem: one N = 64 MMA per tap (K = 16 is one K step), A shifted by the tap's row offset, all nine accumulating in D.
// Ring group ky holds the taps 3 ky .. 3 ky + 2 (2 KB each).
template <int W8, int Q>
__device__ __forceinline__ void issue_tile_stem(bool issuer, uint32_t a_lo_tile, uint32_t b_lo_base, uint32_t d_tmem, bool first_tile,
                                                bool last_tile, uint32_t w_par, uint32_t bar_base) {
  constexpr uint32_t DESC_HI = (128u >> 4) | (1u << 14);
  constexpr uint32_t IDESC = make_idesc(64);
#pragma unroll
  for (int ky = 0; ky < 3; ++ky) {
    if (first_tile) {
      mbar_wait(bar_base + (uint32_t)ky * 8u, w_par);
      tc_fence_after();
    }
    if (issuer) {
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const uint32_t a_lo = a_lo_tile + (uint32_t)((ky - 1) * W8 + (kx - 1));
        const uint32_t b_lo = (b_lo_base + (uint32_t)(3 * ky) * (SLOT_BYTES >> 4) + (uint32_t)kx * (2048u >> 4)) | (64u << 16);
        umma_f16(d_tmem, ((uint64_t)DESC_HI << 32) | a_lo, ((uint64_t)DESC_HI << 32) | b_lo, IDESC, (ky | kx) != 0);
      }
      if (last_tile) umma_commit(bar_base + (uint32_t)(N_SLOTS + ky) * 8u);
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------------
// shared memory plan
// ---------------------------------------------------------------------------------------------------
template <class G>
struct Smem {
  using Ge = Geo<G>;
  static constexpr int ACT_BYTES = 8 * Ge::Q * 16;                 // 69,632
  static constexpr int OFF_ACT0 = 0;
  static constexpr int OFF_ACT1 = ACT_BYTES;
  static constexpr int OFF_W = 2 * ACT_BYTES;                      // 9 x 8 KB weight ring
  static constexpr int OFF_BIAS = OFF_W + N_SLOTS * SLOT_BYTES;    // 10 x 64 f32
  static constexpr int OFF_LOGITS = OFF_BIAS + (N_LAYERS * 64 + 32) * 4;  // [NB][16] f32 (policy logits, value at [15]); the biases end with the 32 Linear biases
  static constexpr int OFF_PART = OFF_LOGITS + Ge::NB * 16 * 4;    // [NB][ROWS][16] f32 row partials of the Linear layers
  static constexpr int OFF_STATES = OFF_PART + 8 * Ge::NB * 8 * 4;   // part: [8 warps][NB][8 slots] f32; then [2][NB] PState
  static constexpr int OFF_SLOTS = OFF_STATES + 2 * Ge::NB * 16;   // [2][NB] u32 (states/slots ping-pong per batch)
  static constexpr int OFF_BARS = (OFF_SLOTS + 2 * Ge::NB * 4 + 15) & ~15;
  // barriers: w_full[9], w_empty[9] (one pair per ring group: 3 used), acc_full[2], acc_drained[2], act_ready[4],
  // stage_ready[4], act0_free, batch[2], claim_go, out_ready, out_free
  static constexpr int N_BARS = 2 * N_SLOTS + 4 + 2 * Ge::NT + 1 + 3 + 2;
  static constexpr int OFF_TMEM = OFF_BARS + N_BARS * 8;
  static constexpr int OFF_NB = OFF_TMEM + 16;                     // [4] boards of batch bb (0 = no more batches), [4] = early flag
  static constexpr int TOTAL = OFF_NB + 32;
};
static_assert(Geo<Connect4>::NB <= 32 && Geo<TicTacToe>::NB <= 32, "one stager lane / one publishing lane per board");

static_assert(Smem<Connect4>::TOTAL <= 232448 && Smem<TicTacToe>::TOTAL <= 232448, "shared memory plan exceeds 227 KB");
// Warp roles.  The eight epilogue warps are warps 4..11 = warpgroups 1 and 2, so that the asynchronous kernel can move
// registers to them with setmaxnreg (a warpgroup-wide instruction); a warp's TMEM lane quadrant is warp % 4.
constexpr int PRODUCER_WARP = 0, MMA_WARP = 1, STAGER_WARP = 2, SPARE_WARP = 3;   // warp 3: publisher of the results
constexpr int EPI_WARP0 = 4, N_EPI_WARPS = 8;
constexpr int THREADS = 32 * (EPI_WARP0 + N_EPI_WARPS);   // 384: static work list (spb_predict, lock-step pipeline)
// asynchronous pipeline: tree warps that share the CTA (and the SM's idle issue slots): warps 12..15 (one warpgroup), 512
// threads = 4 warpgroups x 128 registers = the whole register file.  setmaxnreg moves registers inside what the CTA was given
// at launch (threads x registers per thread): the budgets of a configuration must sum to at most that, not to the register
// file (a tic-tac-toe configuration with 8 tree warps, 640 threads x 96 registers, hung at 72 / 144 / 64 = 62,464 > 61,440 and
// ran 18 % slower than this one at 72 / 136 / 64: the tree code spills at 64 registers).
template <class G> struct RingCfg { static constexpr int TREE_WARPS = 4, REGS_LAUNCH = 128, REGS_LIGHT = 72, REGS_TREE = 96, REGS_EPILOGUE = 168; };
template <class G> constexpr int threads_ring() { return THREADS + 32 * RingCfg<G>::TREE_WARPS; }
template <class G> constexpr bool ring_budget_ok() {
  return 128 * RingCfg<G>::REGS_LIGHT + 256 * RingCfg<G>::REGS_EPILOGUE + 32 * RingCfg<G>::TREE_WARPS * RingCfg<G>::REGS_TREE <= threads_ring<G>() * RingCfg<G>::REGS_LAUNCH &&
         threads_ring<G>() * RingCfg<G>::REGS_LAUNCH <= 65536;
}
static_assert(ring_budget_ok<Connect4>() && ring_budget_ok<TicTacToe>(), "setmaxnreg budget exceeds the CTA's launch allocation");
// setmaxnreg budget of the asynchronous kernel: warpgroup 0 (producer, MMA issuer, stager, one idle warp) and warpgroup 3
// (tree warps) give registers to warpgroups 1 and 2 (epilogue): 128 x 72 + 128 x 96 + 256 x 168 = 64,512 <= 65,536.
constexpr uint32_t CLAIM_GRACE_NS = 4000;   // a batch waits this long for tickets behind its first filled one

// Static work source (spb_predict, lock-step pipeline).  The asynchronous pipeline reads T.leaf_state / writes T.eval_out.
struct EvalWork {
  const PState* states;
  const uint32_t* list;
  const uint32_t* count_dev;
  uint32_t max_n;
  float* out;
  int stride;
  float* logits_out;
};

#ifdef SPB_TRACE
// trace build only (make VARIANT=-DSPB_TRACE): time stamps of CTA 0, plain stores (no read-modify-write), so the
// timeline is that of the production kernel
__device__ unsigned long long g_trace[4][512];   // [0] MMA issue begin, [1] MMA issue end, [2] epilogue body begin, [3] body end; index (b*10+l)*4+t
#define TRACE_B0 (RING ? 300u : 0u)   // asynchronous pipeline: a window of batches in the steady state
#define TRACE(k, b, l, t) do { if (blockIdx.x == 0 && (b) >= TRACE_B0 && (b) < TRACE_B0 + 12u) g_trace[k][((((b) - TRACE_B0) * 10 + (l)) * 4 + (t))] = clock64(); } while (0)
__device__ unsigned long long g_trace_stager[16][4];   // per traced batch: claim begin, claim end, act0_free seen, staged
__device__ unsigned long long g_eval_times[64][4];   // globaltimer: [launch][entry, after griddepcontrol.wait, exit] of CTA 0
__device__ unsigned int g_eval_idx = 0;
__device__ __forceinline__ unsigned long long gtimer() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define TRACE_ST(b, i) do { if (blockIdx.x == 0 && lane == 0 && (b) >= TRACE_B0 && (b) < TRACE_B0 + 12u) g_trace_stager[(b) - TRACE_B0][i] = clock64(); } while (0)
#define TRACE2(i) do { if (blockIdx.x == 0 && bb == TRACE_B0 && lane == 0) g_trace[3][480 + (warp == EPI_WARP0 ? 0 : 8) + (i)] = clock64(); } while (0)
#define TRACE3(i) do { if (blockIdx.x == 0 && bb == TRACE_B0 + 2u && l == 4 && t == 1 && lane == 0 && (warp == EPI_WARP0 || warp == EPI_WARP0 + 4)) g_trace[3][496 + (warp == EPI_WARP0 ? 0 : 8) + (i)] = clock64(); } while (0)
#else
#define TRACE3(i) ((void)0)
#define TRACE2(i) ((void)0)
#define TRACE(k, b, l, t) ((void)0)
#define TRACE_ST(b, i) ((void)0)
#endif

template <class G, bool RING>
__global__ void __launch_bounds__(RING ? threads_ring<G>() : THREADS, 1)
k_eval_umma(const uint8_t* __restrict__ image, const EvalWork W, const Trees T, const AsyncCtl C) {
  using Ge = Geo<G>;
  using Sm = Smem<G>;
  extern __shared__ __align__(1024) uint8_t smem[];
  const PState* __restrict__ states = RING ? T.leaf_state : W.states;
  const uint32_t* __restrict__ list = W.list;
  float* __restrict__ out = RING ? T.eval_out : W.out;
  const int stride = RING ? G::EVAL_STRIDE : W.stride;
  float* __restrict__ logits_out = RING ? nullptr : W.logits_out;
  // Programmatic dependent launch: this grid may start while the tree-step kernel that produces its work list is
  // still running.  Everything up to griddepcontrol.wait touches only shared memory, TMEM and the (static) weight
  // image; the work list, its length and the leaf states are read after the wait.
#ifdef SPB_TRACE
  const unsigned long long tr_entry = gtimer();
#endif
  asm volatile("griddepcontrol.launch_dependents;");
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t s_base = smem_u32(smem);
  const uint32_t bar_base = s_base + Sm::OFF_BARS;
  auto bar_w_full = [&](int s) { return bar_base + (uint32_t)s * 8u; };
  auto bar_w_empty = [&](int s) { return bar_base + (uint32_t)(N_SLOTS + s) * 8u; };
  // Accumulators: two sets of 192 TMEM columns (D | E | F = centre | right | left taps; set s at column 256 s).  The tiles
  // of a CTA form one sequence (batch, layer, tile); tile number g accumulates in set g & 1.  acc_full[s]: the MMAs of the
  // tile in set s have completed (tcgen05.commit); acc_drained[s]: the epilogue warps have read the set (one arrival per
  // warp), the tile after next may overwrite it.  The stem of batch b+1 follows the head conv of batch b in the same
  // sequence, so it runs on the tensor pipe while the epilogue warps are still busy with batch b's head.
  constexpr uint32_t BAR0 = 2 * N_SLOTS;
  auto bar_acc_full = [&](uint32_t set) { return bar_base + (BAR0 + set) * 8u; };
  auto bar_acc_drained = [&](uint32_t set) { return bar_base + (BAR0 + 2u + set) * 8u; };
  auto bar_act_ready = [&](int t) { return bar_base + (BAR0 + 4u + (uint32_t)t) * 8u; };
  // separate barrier for the staged input of a batch: it may complete while act_ready's previous phase is still
  // being consumed by the MMA warp (an mbarrier must never run two phases ahead of a waiter)
  auto bar_stage_ready = [&](int t) { return bar_base + (BAR0 + 4u + (uint32_t)Ge::NT + (uint32_t)t) * 8u; };
  // activation buffer 0 is free for the next batch's input once every MMA of layer 8 has completed (committed by the MMA warp)
  const uint32_t bar_act0_free = bar_base + (BAR0 + 4u + 2u * (uint32_t)Ge::NT) * 8u;
  // batch descriptors: the stager decides how many boards batch bb has (0 = no more batches), writes s_nb[bb & 3] and
  // completes bar_batch[bb & 1]; the producer, the MMA warp and the epilogue warps pick the batch up from there
  auto bar_batch = [&](uint32_t bb) { return bar_base + (BAR0 + 5u + 2u * (uint32_t)Ge::NT + (bb & 1u)) * 8u; };
  // asynchronous pipeline: the MMA warp arrives when it starts layer 7 of a batch — time for the stager to claim the next
  // batch's leaves from the ring (late enough not to hoard leaves, early enough to have them staged behind the head conv)
  const uint32_t bar_claim_go = bar_base + (BAR0 + 7u + 2u * (uint32_t)Ge::NT) * 8u;
  // results of a batch (softmax probabilities + value per board, in s_logits) handed from the epilogue warps to the
  // publisher warp, which writes them to global memory and (asynchronous pipeline) pushes the trees to the ready ring
  const uint32_t bar_out_ready = bar_base + (BAR0 + 8u + 2u * (uint32_t)Ge::NT) * 8u;
  const uint32_t bar_out_free = bar_base + (BAR0 + 9u + 2u * (uint32_t)Ge::NT) * 8u;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + Sm::OFF_TMEM);
  volatile uint32_t* s_nb = reinterpret_cast<volatile uint32_t*>(smem + Sm::OFF_NB);

  // ---- one-time setup -----------------------------------------------------------------------------
  {
    uint4 z = make_uint4(0, 0, 0, 0);
    uint4* p = reinterpret_cast<uint4*>(smem);
    for (int i = tid; i < 2 * Sm::ACT_BYTES / 16; i += (int)blockDim.x) p[i] = z;   // pad rows stay zero forever
    const float* gb = reinterpret_cast<const float*>(image + OFF_BIAS);
    float* sb = reinterpret_cast<float*>(smem + Sm::OFF_BIAS);
    for (int i = tid; i < N_LAYERS * 64; i += (int)blockDim.x) sb[i] = gb[i];
    if (tid < 32) sb[N_LAYERS * 64 + tid] = reinterpret_cast<const float*>(image + off_fcb<G>())[tid];
  }
  if (tid == 0) {
    for (int s = 0; s < N_SLOTS; ++s) { mbar_init(bar_w_full(s), 1); mbar_init(bar_w_empty(s), 1); }
    for (uint32_t set = 0; set < 2; ++set) { mbar_init(bar_acc_full(set), 1); mbar_init(bar_acc_drained(set), N_EPI_WARPS); }
    for (int t = 0; t < Ge::NT; ++t) { mbar_init(bar_act_ready(t), N_EPI_WARPS); mbar_init(bar_stage_ready(t), 32); }
    mbar_init(bar_act0_free, 1);
    mbar_init(bar_batch(0), 1); mbar_init(bar_batch(1), 1); mbar_init(bar_claim_go, 1);
    mbar_init(bar_out_ready, 1); mbar_init(bar_out_free, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == MMA_WARP) tmem_alloc(smem_u32(tmem_slot), 512);
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  asm volatile("griddepcontrol.wait;" ::: "memory");              // the producer grid has completed and its writes are visible
#ifdef SPB_TRACE
  const unsigned long long tr_wait = gtimer();
#endif
  // static work source: this CTA's share of the list, in batches of NB boards
  const uint32_t n_total = RING ? 0u : min(__ldcg(W.count_dev), W.max_n);
  const uint32_t cta = blockIdx.x, ncta = gridDim.x;
  const uint32_t my_begin = (uint32_t)(((uint64_t)n_total * cta) / ncta);
  const uint32_t my_end = (uint32_t)(((uint64_t)n_total * (cta + 1)) / ncta);
  auto wait_batch = [&](uint32_t bb) -> uint32_t {                  // boards of batch bb; 0 = no more batches
    mbar_wait(bar_batch(bb), (bb >> 1) & 1u);
    return s_nb[bb & 3u];
  };

  // Asynchronous kernel: register reallocation by whole warpgroups (setmaxnreg), first thing in every role's branch so
  // that the role's code is compiled for its own budget: the epilogue warps hold two accumulator halves, the skip
  // connection and the layer's biases in registers; the other roles are light.
#define SPB_REGS_LIGHT() do { if (RING) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(RingCfg<G>::REGS_LIGHT)); } while (0)
#define SPB_REGS_TREE() do { if (RING) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(RingCfg<G>::REGS_TREE)); } while (0)
#define SPB_REGS_EPILOGUE() do { if (RING) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(RingCfg<G>::REGS_EPILOGUE)); } while (0)

  if (warp == PRODUCER_WARP) {
    // ===== weight producer: streams the layers' kernel-row blocks into the 3-group ring ==================
    SPB_REGS_LIGHT();
    if (lane == 0) {
      uint32_t use = 0;                                           // completed fills of every slot
      for (uint32_t b = 0; wait_batch(b) != 0u; ++b) {
        for (int l = 0; l < N_LAYERS; ++l) {
          const uint32_t bytes = (uint32_t)layer_tap_bytes(l);
          const uint8_t* src = image + layer_offset(l);
          for (int g = 0; g < 3; ++g) {                            // one ring group (3 slots) and one full/empty barrier pair per kernel row
            if (use > 0) mbar_wait(bar_w_empty(g), (use - 1) & 1u);
            mbar_expect_tx(bar_w_full(g), 3 * bytes);
            bulk_g2s(s_base + Sm::OFF_W + (uint32_t)(3 * g) * SLOT_BYTES, src + (size_t)(3 * g) * bytes, 3 * bytes, bar_w_full(g));
          }
          ++use;
        }
      }
    }
  } else if (warp == MMA_WARP) {
    // ===== MMA issuer ===============================================================================
    SPB_REGS_LIGHT();
    // The whole warp runs the (warp-uniform) control flow so that descriptors stay in uniform registers;
    // one fixed lane issues the tcgen05 instructions.
    {
      const bool issuer = elect_one();
      const uint32_t b_lo_base = ((s_base + Sm::OFF_W) >> 4);
      uint32_t use = 0;        // layer-uses of the weight ring so far
      uint32_t act_par = 0;    // bit t: parity of the next completion of act_ready[t]
      uint32_t stage_par = 0;  // same for stage_ready[t]
      uint32_t g = 0;          // tiles issued so far: tile g accumulates in TMEM set g & 1
      for (uint32_t b = 0;; ++b) {
        const uint32_t nb = wait_batch(b);
        if (nb == 0u) break;
        const int nt = (int)((nb * Ge::BS + 127) / 128);
        for (int l = 0; l < N_LAYERS; ++l) {
          if (RING && l == 7 && issuer) mbar_arrive(bar_claim_go);
          const uint32_t in_buf = s_base + ((l == 0 || (l >= 2 && (l & 1) == 0)) ? Sm::OFF_ACT0 : Sm::OFF_ACT1);
          const uint32_t a_lo_base = ((in_buf >> 4) + Ge::LEAD) | ((uint32_t)Ge::Q << 16);
          const uint32_t cur_par = (l == 0) ? stage_par : act_par;
          if (l == 0) stage_par ^= (1u << nt) - 1u; else act_par ^= (1u << nt) - 1u;
          for (int t = 0; t < nt; ++t, ++g) {
            // A tile's MMAs read its own rows, the last rows of tile t-1 (top kernel row) and the first rows of tile
            // t+1 (bottom kernel row).  Stem: the stager releases tiles in order, wait for tile t+1 up front.  Other
            // layers: wait for tile t (tile 0 only — later tiles were covered by the previous tile's mid-wait) and let
            // the top and middle kernel rows run while the epilogue finishes tile t+1; short batches need that overlap.
            uint32_t mid_bar = 0, mid_par = 0;
            if (l == 0) {
              const int wt = min(t + 1, nt - 1);
              mbar_wait(bar_stage_ready(wt), (cur_par >> wt) & 1u);
            } else {
              if (t == 0) mbar_wait(bar_act_ready(0), cur_par & 1u);
              if (t + 1 < nt) { mid_bar = bar_act_ready(t + 1); mid_par = (cur_par >> (t + 1)) & 1u; }
            }
            const uint32_t set = g & 1u, u = g >> 1;
            if (u > 0u) mbar_wait(bar_acc_drained(set), (u - 1u) & 1u);   // the tile before last has been read out of this set
            tc_fence_after();
            if (lane == 0) TRACE(0, b, l, t);
            const uint32_t a_lo_tile = a_lo_base + (uint32_t)t * 128u;
            const uint32_t d_tmem = tmem_base + set * 256u;
            const bool first = (t == 0), last = (t == nt - 1);
            if (l == 0)
              issue_tile_stem<Ge::W8, Ge::Q>(issuer, a_lo_tile, b_lo_base, d_tmem, first, last, use & 1u, bar_base);
            else if (l < 9)
              issue_tile_triple<Ge::W8, Ge::Q, 4, 192>(issuer, a_lo_tile, b_lo_base, d_tmem, first, last, use & 1u, bar_base, mid_bar, mid_par);
            else
              issue_tile_triple<Ge::W8, Ge::Q, 4, 3 * HEAD_N>(issuer, a_lo_tile, b_lo_base, d_tmem, first, last, use & 1u, bar_base, mid_bar, mid_par);
            if (issuer) {
              umma_commit(bar_acc_full(set));
              if (l == 8 && last) umma_commit(bar_act0_free);
            }
            __syncwarp();
            if (lane == 0) TRACE(1, b, l, t);
          }
          ++use;
        }
      }
    }
  } else if (warp == STAGER_WARP) {
    // ===== stager: fetches the states of batch bb and writes their encoding (get_encoding, connect_four.rs:242-259:
    // channels 0,1,2 of chunk 0; chunk 1 = 0) into activation buffer 0, then releases the stem MMAs.  It runs one
    // batch ahead of the epilogue warps: the global loads are issued before it waits for buffer 0 to be free, and the
    // stem of batch bb can start while the epilogue warps are still busy with the heads of batch bb-1.
    SPB_REGS_LIGHT();
    PState* s_states = reinterpret_cast<PState*>(smem + Sm::OFF_STATES);
    uint32_t* s_slots = reinterpret_cast<uint32_t*>(smem + Sm::OFF_SLOTS);
    Spin sp;
    if (RING) sp.init(C, *C.n_active);
    unsigned long long st_batches = 0, st_boards = 0, st_wait = 0;
    LeafClaimer lc;
    for (uint32_t bb = 0;; ++bb) {
      uint32_t nb = 0;
      PState st_mine = PState{};
      uint32_t slot_mine = 0;
      if (RING) {
        // asynchronous pipeline: claim the batch from the leaf ring once the previous batch has reached layer 7
        if (bb > 0) mbar_wait_backoff<64>(bar_claim_go, (bb - 1) & 1u);
        const unsigned long long tw0 = gtime_ns();
        TRACE_ST(bb, 0);
        nb = claim_batch(C, lc, ncta, (uint32_t)Ge::NB, CLAIM_GRACE_NS, sp, lane, &slot_mine);
        if (nb) { st_wait += gtime_ns() - tw0; ++st_batches; st_boards += nb; }
        TRACE_ST(bb, 1);
      } else {
        const uint32_t b0 = my_begin + bb * Ge::NB;
        nb = b0 < my_end ? min((uint32_t)Ge::NB, my_end - b0) : 0u;
        if ((uint32_t)lane < nb) slot_mine = list ? __ldcg(list + b0 + lane) : (b0 + lane);
      }
      if (lane == 0) {
        s_nb[bb & 3u] = nb;
        mbar_arrive(bar_batch(bb));
      }
      if (nb == 0u) {
        if (RING && lane == 0) {
          atomicAdd(&C.stats[ASTAT_BATCHES], st_batches);
          atomicAdd(&C.stats[ASTAT_BOARDS], st_boards);
          atomicAdd(&C.stats[ASTAT_CLAIM_WAIT_NS], st_wait);
          atomicAdd(&C.stats[ASTAT_EVAL_CTAS], 1ull);
        }
        break;
      }
      const int nt = (int)((nb * Ge::BS + 127) / 128);
      if ((uint32_t)lane < nb) {                                  // written by another grid / another SM: read at L2
        const ulonglong2 raw = __ldcg(reinterpret_cast<const ulonglong2*>(states + slot_mine));
        st_mine.x = raw.x; st_mine.o = raw.y;
      }
      if (bb > 0) mbar_wait_backoff<64>(bar_act0_free, (bb - 1) & 1u);
      TRACE_ST(bb, 2);
      PState* st_buf = s_states + (bb & 1u) * Ge::NB;
      if ((uint32_t)lane < nb) { s_slots[(bb & 1u) * Ge::NB + lane] = slot_mine; st_buf[lane] = st_mine; }
      __syncwarp();
      for (int t = 0; t < nt; ++t) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int m = t * 128 + q * 32 + lane;
          const int bi = m / Ge::BS, rem = m % Ge::BS, r = rem / Ge::W8, c = rem % Ge::W8;
          uint4 v0 = make_uint4(0, 0, 0, 0);
          if ((uint32_t)bi < nb && r < G::ROWS && c < G::COLS) {
            const PState st = st_buf[bi];
            const float e0 = G::encode_cell(st, 0, r, c), e1 = G::encode_cell(st, 1, r, c), e2 = G::encode_cell(st, 2, r, c);
            v0.x = pack_bf16x2(e0, e1);
            v0.y = pack_bf16x2(e2, 0.0f);
          }
          *reinterpret_cast<uint4*>(smem + Sm::OFF_ACT0 + (size_t)(Ge::LEAD + m) * 16) = v0;
          *reinterpret_cast<uint4*>(smem + Sm::OFF_ACT0 + (size_t)Ge::Q * 16 + (size_t)(Ge::LEAD + m) * 16) = make_uint4(0, 0, 0, 0);
        }
        fence_async_smem();
        mbar_arrive(bar_stage_ready(t));
      }
      TRACE_ST(bb, 3);
    }
  } else if (warp >= EPI_WARP0 && warp < EPI_WARP0 + N_EPI_WARPS) {
    // ===== epilogue warps (8 warps, 256 threads): per-layer epilogues, heads =============================
    // Two warps share a TMEM lane quadrant (a tile row) and split the 64 output channels in halves.
    SPB_REGS_EPILOGUE();
    const int et = tid - 32 * EPI_WARP0;                           // 0..255
    const int quad = warp & 3;                                     // TMEM lanes [32*quad, 32*quad+32)
    const int half = (warp - EPI_WARP0) >> 2;                      // channels [32*half, 32*half+32)
    const int row_in_tile = quad * 32 + lane;
    const float* s_bias = reinterpret_cast<const float*>(smem + Sm::OFF_BIAS);
    float* s_logits = reinterpret_cast<float*>(smem + Sm::OFF_LOGITS);
    uint32_t* s_slots = reinterpret_cast<uint32_t*>(smem + Sm::OFF_SLOTS);
    const float* g_wp = reinterpret_cast<const float*>(image + OFF_WP);
    const float* g_wv = reinterpret_cast<const float*>(image + off_wv<G>());
    uint32_t eg = 0;                                               // tiles read so far: tile eg sits in TMEM set eg & 1 (the MMA warp's sequence)

    // Epilogue of conv layer l (0 = stem .. 8) of batch bb: accumulators -> +bias (+skip) -> ReLU -> bf16 -> the other
    // activation buffer, tile by tile; each finished tile releases the next layer's MMAs.
    auto conv_epilogue = [&](uint32_t bb, int l, int t_begin = 0, int t_end = Ge::NT) {
      const uint32_t nb = s_nb[bb & 3u];
      const int nt = min((int)((nb * Ge::BS + 127) / 128), t_end);
      const bool in0 = (l == 0 || (l >= 2 && (l & 1) == 0));
      uint8_t* dst_buf = smem + (in0 ? Sm::OFF_ACT1 : Sm::OFF_ACT0);
      const bool has_skip = (l >= 2 && (l & 1) == 0);              // second conv of a residual block
      const bool stash_skip = (l & 1) == 0 && l <= 6;               // the stem and the blocks' second convs produce a block input x
      float bias_r[32];                                             // this thread's 32 output channels, once per layer: a broadcast
#pragma unroll                                                      // LDS.128 costs two wavefronts of the pipe that bounds this kernel
      for (int q = 0; q < 8; ++q) {
        const float4 bv = *reinterpret_cast<const float4*>(s_bias + l * 64 + half * 32 + q * 4);
        bias_r[4 * q] = bv.x; bias_r[4 * q + 1] = bv.y; bias_r[4 * q + 2] = bv.z; bias_r[4 * q + 3] = bv.w;
      }
      for (int t = t_begin; t < nt; ++t, ++eg) {
        const int m = t * 128 + row_in_tile;
        const int bi = m / Ge::BS, rem = m % Ge::BS, r = rem / Ge::W8, c = rem % Ge::W8;
        const bool valid = (uint32_t)bi < nb && r < G::ROWS && c < G::COLS;
        uint8_t* drow = dst_buf + (size_t)(half * 4) * Ge::Q * 16 + (size_t)(Ge::LEAD + m) * 16;   // chunk 4*half
        const uint32_t set = eg & 1u;
        TRACE3(0);
        mbar_wait(bar_acc_full(set), (eg >> 1) & 1u);
        tc_fence_after();
        if (et == 0) TRACE(2, bb, l, t);
        TRACE3(1);
        // out[r] = D[r] + E[r+1] + F[r-1]: the right tap was computed one row early, the left tap one row late.  Rows
        // 32k-1 are pad cells: lane 31 never needs E of the next warp (its output is a pad cell) and lane 0 takes F = 0
        // (F of a pad-column row is a sum over pad-column cells, which are zero).
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + set * 256u + (uint32_t)half * 32u;
        uint32_t a[32], e[32], f[32];
        tmem_ld16(taddr, a);
        tmem_ld16(taddr + 16u, a + 16);
        if (l != 0) {                                                // the stem accumulates all nine taps in D
          tmem_ld16(taddr + 64u, e);
          tmem_ld16(taddr + 80u, e + 16);
          tmem_ld16(taddr + 128u, f);
          tmem_ld16(taddr + 144u, f + 16);
        }
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_acc_drained(set));           // the tile after next may accumulate in this set
        TRACE3(2);
        float v[32];
#pragma unroll
        for (int q = 0; q < 32; q += 2) {                           // packed f32x2 adds: two channels per instruction
          if (l == 0) { v[q] = __uint_as_float(a[q]); v[q + 1] = __uint_as_float(a[q + 1]); continue; }
          const float e0 = __uint_as_float(__shfl_down_sync(0xffffffffu, e[q], 1)), e1 = __uint_as_float(__shfl_down_sync(0xffffffffu, e[q + 1], 1));
          const float f0 = __uint_as_float(__shfl_up_sync(0xffffffffu, f[q], 1)), f1 = __uint_as_float(__shfl_up_sync(0xffffffffu, f[q + 1], 1));
          v[q] = __uint_as_float(a[q]); v[q + 1] = __uint_as_float(a[q + 1]);
          add2(v[q], v[q + 1], e0, e1);
          if (lane != 0) add2(v[q], v[q + 1], f0, f1);
        }
        TRACE3(3);
        // The skip connection (x + f(x)).relu(), model/mod.rs:163, comes from TMEM: the epilogue that produced x (the stem
        // or the previous block's second conv) left this thread's 32 channels, as stored (bf16 pairs), in the 16 spare
        // columns of an accumulator set — no shared-memory read on the pipe the tensor core needs.
        const uint32_t skaddr = tmem_base + ((uint32_t)(quad * 32) << 16) + ((t & 1) ? 448u : 192u) + (uint32_t)(t >> 1) * 32u + (uint32_t)half * 16u;
        uint32_t sk[16];
        if (has_skip) tmem_ld16(skaddr, sk);
#pragma unroll
        for (int q = 0; q < 32; q += 2) add2(v[q], v[q + 1], bias_r[q], bias_r[q + 1]);
        if (has_skip) {
          tmem_ld_wait();
#pragma unroll
          for (int q = 0; q < 16; ++q) add2(v[2 * q], v[2 * q + 1], bf_lo(sk[q]), bf_hi(sk[q]));
        }
        uint32_t o[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) o[q] = valid ? pack_relu_bf16x2(v[2 * q], v[2 * q + 1]) : 0u;
#pragma unroll
        for (int j = 0; j < 4; ++j)                                 // one 8-channel chunk = one 16-B store
          *reinterpret_cast<uint4*>(drow + (size_t)j * Ge::Q * 16) = make_uint4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
        if (stash_skip) { tmem_st16(skaddr, o); tmem_st_wait(); }   // this layer's output is the next block's x
        TRACE3(4);
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_act_ready(t));
        TRACE3(5);
        if (et == 0) TRACE(3, bb, l, t);
      }
    };

    // Epilogue of the fused head conv of batch bb: ReLU(policy conv) channels 0..31 and ReLU(value conv) channels
    // 32..34 go, as bf16, to the dead chunks 2..6 of activation buffer 0 (chunks 0,1 hold the next batch's input;
    // layer 1 rewrites every chunk before buffer 0 is read as an operand again).
    auto head_epilogue = [&](uint32_t bb) {
      const uint32_t nb = s_nb[bb & 3u];
      const int nt = (int)((nb * Ge::BS + 127) / 128);
      const float* bias = s_bias + 9 * 64;
      for (int t = 0; t < nt; ++t, ++eg) {
        const int m = t * 128 + row_in_tile;
        const int bi = m / Ge::BS, rem = m % Ge::BS, r = rem / Ge::W8, c = rem % Ge::W8;
        const bool valid = (uint32_t)bi < nb && r < G::ROWS && c < G::COLS;
        const uint32_t set = eg & 1u;
        mbar_wait(bar_acc_full(set), (eg >> 1) & 1u);
        tc_fence_after();
        if (et == 0) TRACE(2, bb, 9, t);
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + set * 256u;
        // columns [0,48) = D (centre taps), [48,96) = E (right taps, one row early), [96,144) = F (left taps, one row late)
        uint32_t a[16], av[4], e[16], ev[4], f[16], fv[4];
        tmem_ld16(taddr + (uint32_t)half * 16u, a);
        tmem_ld16(taddr + (uint32_t)HEAD_N + (uint32_t)half * 16u, e);
        tmem_ld16(taddr + 2u * (uint32_t)HEAD_N + (uint32_t)half * 16u, f);
        if (half == 1) { tmem_ld4(taddr + 32u, av); tmem_ld4(taddr + (uint32_t)HEAD_N + 32u, ev); tmem_ld4(taddr + 2u * (uint32_t)HEAD_N + 32u, fv); }
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_acc_drained(set));
#pragma unroll
        for (int q = 0; q < 16; ++q) {
          const float e1 = __uint_as_float(__shfl_down_sync(0xffffffffu, e[q], 1));
          const float f1 = __uint_as_float(__shfl_up_sync(0xffffffffu, f[q], 1));
          float v = __uint_as_float(a[q]) + e1;
          if (lane != 0) v += f1;
          a[q] = __float_as_uint(v);
        }
        if (half == 1) {                                            // warp-uniform: half is a property of the warp
#pragma unroll
          for (int q = 0; q < 3; ++q) {
            const float e1 = __uint_as_float(__shfl_down_sync(0xffffffffu, ev[q], 1));
            const float f1 = __uint_as_float(__shfl_up_sync(0xffffffffu, fv[q], 1));
            av[q] = __float_as_uint((__uint_as_float(av[q]) + e1) + (lane == 0 ? 0.0f : f1));
          }
        }
        if (valid) {
          uint8_t* prow = smem + Sm::OFF_ACT0 + (size_t)(Ge::LEAD + m) * 16;
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            uint4 o;
            const float* bj = bias + half * 16 + j * 8;
            o.x = pack_bf16x2(fmaxf(__uint_as_float(a[j * 8 + 0]) + bj[0], 0.f), fmaxf(__uint_as_float(a[j * 8 + 1]) + bj[1], 0.f));
            o.y = pack_bf16x2(fmaxf(__uint_as_float(a[j * 8 + 2]) + bj[2], 0.f), fmaxf(__uint_as_float(a[j * 8 + 3]) + bj[3], 0.f));
            o.z = pack_bf16x2(fmaxf(__uint_as_float(a[j * 8 + 4]) + bj[4], 0.f), fmaxf(__uint_as_float(a[j * 8 + 5]) + bj[5], 0.f));
            o.w = pack_bf16x2(fmaxf(__uint_as_float(a[j * 8 + 6]) + bj[6], 0.f), fmaxf(__uint_as_float(a[j * 8 + 7]) + bj[7], 0.f));
            *reinterpret_cast<uint4*>(prow + (size_t)(2 + half * 2 + j) * Ge::Q * 16) = o;
          }
          if (half == 1) {
            uint4 o = make_uint4(0, 0, 0, 0);
            o.x = pack_bf16x2(fmaxf(__uint_as_float(av[0]) + bias[32], 0.f), fmaxf(__uint_as_float(av[1]) + bias[33], 0.f));
            o.y = pack_bf16x2(fmaxf(__uint_as_float(av[2]) + bias[34], 0.f), 0.f);
            *reinterpret_cast<uint4*>(prow + (size_t)6 * Ge::Q * 16) = o;
          }
        }
        if (et == 0) TRACE(3, bb, 9, t);
      }
    };

    // The two Linear layers, softmax (model/mod.rs:63) and tanh (connect_four.rs:71) of batch bb.  A thread owns one
    // unit = (position, 8-channel chunk) of the head activations — 4P policy units, then P value units — and keeps the
    // unit's weights for 8 output slots in registers (slots of pass og: policy outputs og..og+7, the value right after
    // the last policy output).  Per board: ONE 16-byte shared-memory read per thread (the tensor pipe needs the
    // shared-memory bandwidth), 8 slot partials, a 7-shuffle transposing reduction inside the warp, then the 8 warp
    // partials are added in warp order.  The summation order of a board is fixed, whatever the batch looks like.
    // The Linear layers' geometry of this thread: one unit = (position, 8-channel chunk) of the head activations.
    constexpr int LH_P = Ge::P;
    constexpr int NOUT = G::A + 1;
    const bool is_pol = et < 4 * LH_P, is_val = !is_pol && et < 5 * LH_P;
    const int pos = is_pol ? (et % LH_P) : (is_val ? et - 4 * LH_P : 0);
    const int c4 = is_pol ? (et / LH_P) : 4;                         // position-major inside a chunk: conflict-free reads
    // the unit's weights for the 8 output slots og..og+7 (policy outputs, the value right after the last policy output)
    auto load_head_weights = [&](float (&w)[8][8], int og) {
#pragma unroll
      for (int s = 0; s < 8; ++s) {
        const int o = og + s;
#pragma unroll
        for (int j = 0; j < 8; ++j) w[s][j] = 0.0f;
        const float* src = nullptr;
        if (is_pol && o < G::A) src = g_wp + ((size_t)o * LH_P + pos) * NET_POLICY_CH + c4 * 8;
        if (is_val && o == G::A) src = g_wv + pos * 8;
        if (src) {
          const float4 w0 = __ldg(reinterpret_cast<const float4*>(src)), w1 = __ldg(reinterpret_cast<const float4*>(src) + 1);
          w[s][0] = w0.x; w[s][1] = w0.y; w[s][2] = w0.z; w[s][3] = w0.w;
          w[s][4] = w1.x; w[s][5] = w1.y; w[s][6] = w1.z; w[s][7] = w1.w;
        }
      }
    };
    // Board loop of the Linear layers for the output group og (weights w): every warp leaves its partial sums in s_part.
    auto heads_partials = [&](uint32_t bb, float (&w)[8][8], uint32_t bi_begin = 0, uint32_t bi_end = Ge::NB) {   // bi_begin: a multiple of 3
      const uint32_t nb = s_nb[bb & 3u];
      const uint32_t bend = min(nb, bi_end);
      float* s_part = reinterpret_cast<float*>(smem + Sm::OFF_PART);   // [8 warps][NB][8 slots]
      const int we = warp - EPI_WARP0;
      const uint32_t roff = (uint32_t)((is_pol || is_val ? (2 + c4) * Ge::Q * 16 : 0) + ((pos / G::COLS) * Ge::W8 + (pos % G::COLS)) * 16);
      TRACE2(0);
      {
        TRACE2(1);
        const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4;
        // three boards per trip so that the loads, FMA chains and shuffle levels of different boards overlap
        uint4 vn[3];                                                // the next trip's activations, fetched a trip ahead
#pragma unroll
        for (int k = 0; k < 3; ++k)
          vn[k] = *reinterpret_cast<const uint4*>(smem + Sm::OFF_ACT0 + (size_t)(Ge::LEAD + min(bi_begin + (uint32_t)k, nb - 1u) * Ge::BS) * 16 + roff);
        for (uint32_t bi0 = bi_begin; bi0 < bend; bi0 += 3) {
          float sres[3];
          uint4 v[3];
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            v[k] = vn[k];
            vn[k] = *reinterpret_cast<const uint4*>(smem + Sm::OFF_ACT0 + (size_t)(Ge::LEAD + min(bi0 + 3u + (uint32_t)k, nb - 1u) * Ge::BS) * 16 + roff);
          }
          float q[3][4], r2[3][2];
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            const float x0 = bf_lo(v[k].x), x1 = bf_hi(v[k].x), x2 = bf_lo(v[k].y), x3 = bf_hi(v[k].y);
            const float x4 = bf_lo(v[k].z), x5 = bf_hi(v[k].z), x6 = bf_lo(v[k].w), x7 = bf_hi(v[k].w);
            float p[8];
#pragma unroll
            for (int s = 0; s < 8; ++s) {
              float a = x0 * w[s][0];
              a = fmaf(x1, w[s][1], a); a = fmaf(x2, w[s][2], a); a = fmaf(x3, w[s][3], a);
              a = fmaf(x4, w[s][4], a); a = fmaf(x5, w[s][5], a); a = fmaf(x6, w[s][6], a); a = fmaf(x7, w[s][7], a);
              p[s] = a;
            }
            // transposing reduction: 8 slots x 32 lanes -> lane L (L % 4 == 0) holds the warp's sum of slot L / 4
#pragma unroll
            for (int i = 0; i < 4; ++i) q[k][i] = (b4 ? p[i + 4] : p[i]) + __shfl_xor_sync(0xffffffffu, b4 ? p[i] : p[i + 4], 16);
          }
#pragma unroll
          for (int k = 0; k < 3; ++k) {
#pragma unroll
            for (int i = 0; i < 2; ++i) r2[k][i] = (b3 ? q[k][i + 2] : q[k][i]) + __shfl_xor_sync(0xffffffffu, b3 ? q[k][i] : q[k][i + 2], 8);
          }
#pragma unroll
          for (int k = 0; k < 3; ++k) sres[k] = (b2 ? r2[k][1] : r2[k][0]) + __shfl_xor_sync(0xffffffffu, b2 ? r2[k][0] : r2[k][1], 4);
#pragma unroll
          for (int k = 0; k < 3; ++k) sres[k] += __shfl_xor_sync(0xffffffffu, sres[k], 2);
#pragma unroll
          for (int k = 0; k < 3; ++k) sres[k] += __shfl_xor_sync(0xffffffffu, sres[k], 1);
          if ((lane & 3) == 0) {
#pragma unroll
            for (int k = 0; k < 3; ++k)
              if (bi0 + (uint32_t)k < nb) s_part[((size_t)we * Ge::NB + bi0 + k) * 8 + (lane >> 2)] = sres[k];
          }
        }
        TRACE2(2);
      }
    };
    // The 8 warp partials of every (board, slot) are added in warp order: the summation order of a board is fixed.
    auto heads_reduce = [&](uint32_t bb, int og) {
      const uint32_t nb = s_nb[bb & 3u];
      const float* s_part = reinterpret_cast<const float*>(smem + Sm::OFF_PART);
      epi_bar_sync();
      if (og == 0 && bb > 0) mbar_wait(bar_out_free, (bb - 1) & 1u);   // the publisher has read the previous batch's results
      for (int i = et; i < (int)nb * 8; i += 256) {
        const int bi = i >> 3, sl = i & 7, o = og + sl;
        if (o < NOUT) {
          float acc = 0.0f;
#pragma unroll
          for (int wv_ = 0; wv_ < 8; ++wv_) acc += s_part[((size_t)wv_ * Ge::NB + bi) * 8 + sl];
          s_logits[bi * 16 + (o == G::A ? 15 : o)] = acc;
        }
      }
      epi_bar_sync();
      TRACE2(3);
    };
    // softmax (model/mod.rs:63) and tanh (connect_four.rs:71): LG lanes per board, lane a < A owns action a, the last lane
    // of the group the value.  The normaliser is the sum of the exponentials in action order (one lane would produce the
    // same bits).  The board's record (softmax probabilities, value) replaces its logits in s_logits: the publisher warp
    // writes it to global memory, so that the global stores and the release of the trees are not on the epilogue warps' path.
    auto heads_softmax = [&](uint32_t bb) {
      const uint32_t nb = s_nb[bb & 3u];
      constexpr int LG = G::A <= 7 ? 8 : 16;
      const float* fcb = s_bias + N_LAYERS * 64;
      const int a = et % LG;
      for (uint32_t bi = (uint32_t)(et / LG); bi < ((nb + 256 / LG - 1) / (256 / LG)) * (256 / LG); bi += 256 / LG) {   // warp-uniform trip count
        const bool live = bi < nb;
        const float raw = live ? s_logits[bi * 16 + (a == LG - 1 ? 15 : a)] : 0.0f;
        const float lg = (a < G::A) ? raw + fcb[a] : -INFINITY;
        float mx = lg;
#pragma unroll
        for (int o = LG / 2; o >= 1; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        const float ex = (a < G::A) ? expf(lg - mx) : 0.0f;
        float sum = 0.0f;
#pragma unroll
        for (int k = 0; k < G::A; ++k) sum += __shfl_sync(0xffffffffu, ex, (lane & ~(LG - 1)) + k);
        if (live) {
          if (a < G::A) s_logits[bi * 16 + a] = ex / sum;
          else if (a == LG - 1) s_logits[bi * 16 + 15] = tanhf(raw + fcb[16]);
          if (logits_out && a < G::A) logits_out[(size_t)s_slots[(bb & 1u) * Ge::NB + bi] * G::A + a] = lg;   // spb_predict(raw_logits) only
        }
      }
      TRACE2(4);
      epi_bar_sync();                                               // the records are complete
      if (et == 0) mbar_arrive(bar_out_ready);
      TRACE2(5);
    };
    // The two Linear layers, softmax and tanh of batch bb.  w_first: the weights of the first output group.
    auto linear_heads = [&](uint32_t bb, float (&w_first)[8][8]) {
      heads_partials(bb, w_first);
      heads_reduce(bb, 0);
      for (int og = 8; og < NOUT; og += 8) {
        float w[8][8];
        load_head_weights(w, og);
        heads_partials(bb, w);
        heads_reduce(bb, og);
      }
      heads_softmax(bb);
    };

    constexpr uint32_t NOT_YET = 0xFFFFFFFFu;
    uint32_t nb_cur = wait_batch(0);
    if (nb_cur != 0u) conv_epilogue(0, 0);
    bool l1_done = false;                                           // layer 1 of this batch was handled inside the previous batch's heads
    for (uint32_t b = 0; nb_cur != 0u; ++b) {
      for (int l = l1_done ? 2 : 1; l < 9; ++l) conv_epilogue(b, l);
      l1_done = false;
      head_epilogue(b);
      // Has the stager already decided the next batch?  One thread looks, so that all 256 epilogue threads take the
      // same branch (both branches contain named barriers).
      if (et == 0) s_nb[4] = mbar_test(bar_batch(b + 1), ((b + 1) >> 1) & 1u) ? s_nb[(b + 1) & 3u] : NOT_YET;
      epi_bar_sync();                                               // every head activation of the batch is in shared memory
      uint32_t nb_next = s_nb[4];
      float w_heads[8][8];
      if (nb_next != NOT_YET) {
        // The stem of the next batch ran on the tensor pipe behind this batch's head conv (the stager had its input
        // ready): release layer 1 of the next batch before spending time on this batch's Linear layers.
        load_head_weights(w_heads, 0);                              // in flight under the stem's (light: one accumulator, no shuffles) epilogue
        if (nb_next != 0u) conv_epilogue(b + 1, 0);
        if (NOUT <= 8 && nb_next != 0u) {
          // Only the board loop reads the head activations in buffer 0, which layer 1's epilogue overwrites: the reduction,
          // softmax and hand-off to the publisher follow layer 1 of the next batch, whose MMAs would otherwise wait for them
          // (two accumulator sets: the MMA warp is at most two tiles ahead of the epilogue warps).  Interleaving the board
          // loop with layer 1's tiles was tried: the 64 weight registers do not survive the conv epilogue (spills inside
          // the board loop, 81 ms instead of 65 ms per search).
          heads_partials(b, w_heads);
          epi_bar_sync();                                           // every warp has read the head activations: buffer 0 may be overwritten
          conv_epilogue(b + 1, 1);
          l1_done = true;
          heads_reduce(b, 0);
          heads_softmax(b);
        } else {
          linear_heads(b, w_heads);
        }
      } else {
        // The next batch is not known yet (few leaves in flight): its leaves may depend on THIS batch's results, so the
        // results go out first.
        load_head_weights(w_heads, 0);
        linear_heads(b, w_heads);
        nb_next = wait_batch(b + 1);
        if (nb_next != 0u) conv_epilogue(b + 1, 0);
      }
      nb_cur = nb_next;
    }
  }

  if (RING && warp >= EPI_WARP0 + N_EPI_WARPS) {
    // ===== warps 12..15: the tree side of the pipeline (async.cuh) ====================================
    SPB_REGS_TREE();
    tree_worker<G>(T, C, lane);
  } else if (warp == SPARE_WARP) {
    // ===== warp 3: publisher.  Writes the records of a finished batch (out[slot] = softmax probabilities + value) and, in
    // the asynchronous pipeline, hands the evaluated trees to the tree warps through the ready ring. =====================
    SPB_REGS_LIGHT();
    const float* s_logits = reinterpret_cast<const float*>(smem + Sm::OFF_LOGITS);
    const uint32_t* s_slots = reinterpret_cast<const uint32_t*>(smem + Sm::OFF_SLOTS);
    for (uint32_t b = 0;; ++b) {
      const uint32_t nb = wait_batch(b);
      if (nb == 0u) break;
      mbar_wait(bar_out_ready, b & 1u);
      uint32_t slot = 0;
      float rec[G::A + 1];
      if ((uint32_t)lane < nb) {
        slot = s_slots[(b & 1u) * Ge::NB + lane];
#pragma unroll
        for (int a = 0; a < G::A; ++a) rec[a] = s_logits[lane * 16 + a];
        rec[G::A] = s_logits[lane * 16 + 15];
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_out_free);
      if ((uint32_t)lane < nb) {
        float* o = out + (size_t)slot * stride;
#pragma unroll
        for (int a = 0; a <= G::A; ++a) o[a] = rec[a];
      }
      if (RING) ring_push_warp(C.ready, nb, slot, lane);            // each lane releases the record it just wrote
    }
  }

  // ---- teardown -----------------------------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
#ifdef SPB_TRACE
  if (blockIdx.x == 0 && tid == 0) {
    const unsigned int i = g_eval_idx++ & 63u;
    g_eval_times[i][0] = tr_entry; g_eval_times[i][1] = tr_wait; g_eval_times[i][2] = gtimer();
  }
#endif
}

// Per device (one process may drive one engine per GPU from several host threads): SM count + opt-in shared memory.
template <class G, bool RING>
static cudaError_t prepare(int* sm_count_out) {
  static std::mutex mu;
  static int sm_counts[64] = {};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
  std::lock_guard<std::mutex> lock(mu);
  if (sm_counts[dev] == 0) {
    int n = 0;
    e = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_eval_umma<G, RING>, cudaFuncAttributeMaxDynamicSharedMemorySize, Smem<G>::TOTAL);
    if (e != cudaSuccess) return e;
    sm_counts[dev] = n;
  }
  *sm_count_out = sm_counts[dev];
  return cudaSuccess;
}

template <class G>
static cudaError_t launch_t(const Evaluator::DevNet& net, const PState* states, const uint32_t* list, const uint32_t* count_dev,
                            uint32_t max_n, float* out, int stride, float* logits_out, cudaStream_t stream, bool overlap) {
  int sm_count = 0;
  cudaError_t e = prepare<G, false>(&sm_count);
  if (e != cudaSuccess) return e;
  const unsigned grid = (unsigned)std::max(1, std::min<int>(sm_count, (int)max_n));
  // programmatic stream serialization: the kernel may start (set-up only) before the previous kernel in the stream ends
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(THREADS);
  cfg.dynamicSmemBytes = Smem<G>::TOTAL;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = overlap ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  EvalWork W{states, list, count_dev, max_n, out, stride, logits_out};
  return cudaLaunchKernelEx(&cfg, k_eval_umma<G, false>, reinterpret_cast<const uint8_t*>(net.w_umma), W, Trees{}, AsyncCtl{});
}

// Asynchronous pipeline: one resident CTA per SM (evaluator warps + tree warps) for the whole search.
template <class G>
static cudaError_t launch_ring_t(const Evaluator::DevNet& net, const Trees& T, const AsyncCtl& C, cudaStream_t stream) {
  int sm_count = 0;
  cudaError_t e = prepare<G, true>(&sm_count);
  if (e != cudaSuccess) return e;
  const unsigned grid = (unsigned)std::max(1, std::min<int>(sm_count, (int)T.G));
  k_eval_umma<G, true><<<grid, threads_ring<G>(), Smem<G>::TOTAL, stream>>>(reinterpret_cast<const uint8_t*>(net.w_umma), EvalWork{}, T, C);
  return cudaGetLastError();
}

#ifdef SPB_TRACE
extern "C" int spb_debug_eval_times_v2(unsigned long long* out) {
  unsigned int z = 0;
  int rc = (int)cudaMemcpyFromSymbol(out, g_eval_times, sizeof(unsigned long long) * 64 * 4);
  rc |= (int)cudaMemcpyToSymbol(g_eval_idx, &z, sizeof z);
  return rc;
}
extern "C" int spb_debug_trace_stager(unsigned long long* out) { return (int)cudaMemcpyFromSymbol(out, g_trace_stager, sizeof(unsigned long long) * 16 * 4); }
extern "C" int spb_debug_trace_v2(unsigned long long* out, int reset) {
  int rc = (int)cudaMemcpyFromSymbol(out, g_trace, sizeof(unsigned long long) * 4 * 512);
  if (reset) { static unsigned long long z[4 * 512]; rc |= (int)cudaMemcpyToSymbol(g_trace, z, sizeof z); }
  return rc;
}
#endif

cudaError_t launch(const Evaluator::DevNet& net, int game, const PState* states, const uint32_t* list, const uint32_t* count_dev,
                   uint32_t max_n, float* out, int stride, float* logits_out, cudaStream_t stream, bool overlap) {
  if (game == SPB_GAME_CONNECT4) return launch_t<Connect4>(net, states, list, count_dev, max_n, out, stride, logits_out, stream, overlap);
  return launch_t<TicTacToe>(net, states, list, count_dev, max_n, out, stride, logits_out, stream, overlap);
}

cudaError_t launch_ring(const Evaluator::DevNet& net, int game, const Trees& T, const AsyncCtl& C, cudaStream_t stream) {
  if (game == SPB_GAME_CONNECT4) return launch_ring_t<Connect4>(net, T, C, stream);
  return launch_ring_t<TicTacToe>(net, T, C, stream);
}

}  // namespace umma
}  // namespace spb
