// chess_net.cuh — host interface of the chess policy/value network (ref: src/model/chess.rs:50-83 over
// src/model/mod.rs:152-184): 19 -> 256 stem, 10 residual blocks of two 3x3 convs (256 -> 256, BatchNorm folded), policy
// head 1x1 conv 256 -> 256, ReLU, 1x1 conv 256 -> 73 (flattened to 73*8*8 logits), value head 1x1 conv 256 -> 1, ReLU,
// Linear 64 -> 256, ReLU, Linear 256 -> 1, tanh.  1.526 GFLOP per position, 99 % of it in the 20 residual convs.
#pragma once
#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "chess.cuh"

struct spb_chess_engine;

namespace spb {
namespace chess {

constexpr int NET_HIDDEN = 256;        // model/chess.rs:18 num_hidden
constexpr int NET_BLOCKS = 10;         // model/chess.rs:18 num_resnet_blocks
constexpr int NET_CONV3 = 1 + 2 * NET_BLOCKS;
constexpr int NET_IN = SPB_CHESS_PLANES;   // 19
constexpr int NET_MOVE_PLANES = 73;
constexpr float NET_BN_EPS = 1e-5f;

// Folded network on the host.
struct HostNet {
  struct Conv { int oc = 0, ic = 0, k = 0; std::vector<float> w, b; };   // w [oc][ic][k][k]
  Conv conv3[NET_CONV3];            // 0 stem, 1..20 residual convs (BatchNorm folded in)
  Conv p1, p2, vconv;               // 1x1 convs of the heads
  std::vector<float> fc1_w, fc1_b;  // [256][64], [256]
  std::vector<float> fc2_w, fc2_b;  // [1][256], [1]
};
// weights.cu: safetensors (tch VarStore creation-order names or explicit names) -> folded HostNet
bool parse_safetensors_chess(const void* blob, size_t n, HostNet* out, std::string* err);

struct Net;
Net* net_create(uint32_t max_positions, std::string* err);
void net_destroy(Net* net);
bool net_upload(Net* net, const HostNet& host, std::string* err);
bool net_loaded(const Net* net);
void net_set_loaded(Net* net, bool ok);
double net_flops_per_position();

// The weight image net_upload writes, for the device packer (weights_device.cu) and the broadcast (gather.cu).
//   d_w: per 3x3 conv (i < 21; KC32 = 1 for the stem, 8 after) and per policy 1x1 conv (p1: N = 256, p2: N = 80) the
//        stages [kc32][tap][4 chunks][N][8] bf16 of pack_conv, output channels >= OC and input channels >= IC zero; a
//        residual conv run by CTA pairs (res_halves) splits every stage into two halves [rank][4 chunks][N/2][8]
//   d_f: f32 at the offsets below (in floats): folded biases, p1 / p2 biases, the value conv's weights and bias, fc1
//        transposed to [64][256], fc1 bias, fc2 weights and bias; every other float zero
struct NetImage {
  uint8_t* d_w = nullptr;
  size_t w_bytes = 0;
  float* d_f = nullptr;
  size_t f_count = 0;
  size_t off_conv[NET_CONV3] = {}, off_p1 = 0, off_p2 = 0;
  size_t off_bias[NET_CONV3] = {}, off_bp1 = 0, off_bp2 = 0, off_vw = 0, off_vb = 0, off_f1w = 0, off_f1b = 0, off_f2w = 0, off_f2b = 0;
  bool res_halves = false;
};
NetImage net_image(Net* net);

// Evaluates pos[list[i]] (repetition count reps[list[i]] for plane 16) for i < *count_dev (read on the device, at most the
// capacity of activation set `set`: 0 = max_positions, 1 = half of it) and writes logits[list[i]][4672] (raw, f32) and values[list[i]] (tanh).  list == nullptr: identity.
cudaError_t net_forward(Net* net, int set, const Pos* pos, const uint32_t* reps, const uint32_t* list, const uint32_t* count_dev, float* logits,
                        float* values, cudaStream_t stream, uint32_t* launched);
cudaError_t net_time_conv(Net* net, const uint32_t* count_dev, uint32_t iters, cudaStream_t stream, cudaEvent_t ev0, cudaEvent_t ev1, float* avg_ms);
// the evaluator step of the lock-step search: the pending leaves of one range of e->T's trees (work list `list`, its length on
// the device), in activation set `set`, on `stream`
int32_t net_forward_leaves(spb_chess_engine* e, int set, const uint32_t* list, const uint32_t* count_dev, cudaStream_t stream, uint32_t* launched);

}  // namespace chess
}  // namespace spb
