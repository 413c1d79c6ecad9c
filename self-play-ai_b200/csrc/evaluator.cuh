// evaluator.cuh — host interface of the policy/value evaluator (Model::predict's tensor part,
// ref: src/model/mod.rs:60-67,95; architecture ref: src/model/mod.rs:152-184,
// src/model/connect_four.rs:50-81, src/model/tictactoe.rs:50-81).
#pragma once
#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "games.cuh"

namespace spb {

struct Trees;
struct AsyncCtl;

constexpr int NET_HIDDEN = 64;     // model/connect_four.rs:18 num_hidden
constexpr int NET_BLOCKS = 4;      // model/connect_four.rs:18 num_resnet_blocks
constexpr int NET_POLICY_CH = 32;  // model/connect_four.rs:60
constexpr int NET_VALUE_CH = 3;    // model/connect_four.rs:66
constexpr int NET_CONVS = 1 + 2 * NET_BLOCKS + 2;   // stem + 8 residual convs + policy conv + value conv
constexpr float BN_EPS = 1e-5f;    // tch BatchNormConfig default

// Folded network on the host: conv weights [OC][IC][3][3] with BatchNorm (eval mode) folded in.
struct HostNet {
  int game = -1, rows = 0, cols = 0, actions = 0;
  struct Conv { int oc = 0, ic = 0; std::vector<float> w, b; };
  Conv conv[NET_CONVS];            // 0 stem, 1..8 residual, 9 policy conv, 10 value conv
  std::vector<float> pfc_w, pfc_b; // [A][32*R*C], [A]
  std::vector<float> vfc_w, vfc_b; // [1][3*R*C], [1]
};

// Parses a safetensors blob written from the reference's VarStore (or by tests) into a folded HostNet.
// Returns false and fills `err` on malformed input / missing tensors / shape mismatch.
bool parse_safetensors_net(const void* blob, size_t n, int game, HostNet* out, std::string* err);

class Evaluator {
 public:
  Evaluator() = default;
  ~Evaluator();
  Evaluator(const Evaluator&) = delete;
  Evaluator& operator=(const Evaluator&) = delete;

  // Byte offsets of the sections of the weight image of `game` (upload writes them, weights_device.cu packs them on the
  // device): per conv the bf16 weights of the SIMT kernel [OC][IC*9] and the f32 biases, the f32 Linear layers, and the
  // tcgen05 image (umma::image_layout).  Every section starts 256-byte aligned; the gaps are zero.
  struct Layout { size_t wsimt[NET_CONVS], bias[NET_CONVS], pw, pb, vw, vb, umma, bytes = 0; };
  static Layout layout(int game);

  // Uploads the folded net: bf16 conv weights in the tcgen05 shared-memory layout + f32 biases / FCs.
  bool upload(const HostNet& net, std::string* err);
  // The image of `game` to be rewritten in place (the device load, the broadcast of a non-root rank): allocated, and the
  // net marked unloaded, only when there is none of that size yet; nullptr (err set) when out of memory.  The caller marks
  // the net unloaded before it writes and loaded once the image is whole.
  uint8_t* image_for(int game, std::string* err);
  void set_loaded(bool ok) { loaded_ = ok; }
  bool loaded() const { return loaded_; }
  int game() const { return game_; }
  uint8_t* image() const { return static_cast<uint8_t*>(d_blob_); }
  size_t image_bytes() const { return blob_bytes_; }

  // Evaluates states[list[i]] for i < *count_dev (count read on the device; at most max_n) and writes
  // out[list[i]*stride + 0..A) = softmax(logits) (NOT masked), out[list[i]*stride + A] = tanh value.
  // logits_out (nullable) receives raw logits at [list[i]*A + a].  list == nullptr means identity.
  // simt = true selects the CUDA-core cross-check kernel instead of the tcgen05 kernel.
  cudaError_t launch(const PState* states, const uint32_t* list, const uint32_t* count_dev, uint32_t max_n,
                     float* out, int stride, float* logits_out, bool simt, cudaStream_t stream, bool overlap = true);

  // Asynchronous search pipeline (async.cuh): launches the resident evaluator + tree-warp kernel that serves the leaf
  // ring until every tree of the search is done.
  cudaError_t launch_ring(const Trees& T, const AsyncCtl& C, cudaStream_t stream);

  // FLOPs per evaluated position (2*MAC over convs and FCs; SURVEY.md §8a: 26,630,268 for Connect4).
  double flops_per_position() const;

 private:
  void point_at(int game);      // dev_ and the geometry for the image of `game` in d_blob_
  bool loaded_ = false;
  int game_ = -1, rows_ = 0, cols_ = 0, actions_ = 0;
  void* d_blob_ = nullptr;      // one allocation holding everything below
  size_t blob_bytes_ = 0;
 public:
  // device pointers into d_blob_ (public for the kernels' parameter structs)
  struct DevNet {
    const uint16_t* w_simt[NET_CONVS];   // bf16 [OC][IC*9] (k = ic*9 + tap), SIMT kernel
    const float* bias[NET_CONVS];        // f32 [OC]
    const uint16_t* w_umma;              // weight image of the tcgen05 kernel (evaluator_umma.cu: UMMA operand layout)
    const float* pfc_w; const float* pfc_b; const float* vfc_w; const float* vfc_b;
    int rows, cols, actions;
  } dev_{};
};

}  // namespace spb
