// weights.cuh — the name resolver of the checkpoint readers (weights.cu), shared by the safetensors path
// (spb_load_weights, spb_chess_load_weights) and the device-tensor path (weights_device.cu).
//
// A checkpoint is a list of (name, dtype, shape) entries.  The resolver maps them to the network's roles (the explicit
// names, or tch's creation-order census), checks every shape, and hands each role's entry to a `take` callback in the
// order the safetensors reader has always loaded them, so that both paths report the same first error.
#pragma once
#include <cstdint>
#include <functional>
#include <string>
#include <vector>

namespace spb {

struct WeightEntry {
  std::string name;
  std::string dtype;               // safetensors spelling: "F32", "BF16", "F64", "F16", ...
  std::vector<int64_t> shape;
  size_t begin = 0, end = 0;       // data_offsets (safetensors only)
};

// Roles: conv i has the six roles 6i + ROLE_W .. 6i + ROLE_VAR (conv weight and bias, BatchNorm weight, bias, running mean
// and variance); the heads follow the convs.
enum { ROLE_W = 0, ROLE_B, ROLE_G, ROLE_BETA, ROLE_MEAN, ROLE_VAR };
// Connect4 / tic-tac-toe: 11 convs (stem, 8 residual, policy, value), then the two Linear layers
enum { NET_ROLE_PFC_W = 66, NET_ROLE_PFC_B, NET_ROLE_VFC_W, NET_ROLE_VFC_B, NET_ROLES };
// chess: 21 convs, then policy_conv1 / policy_conv2 / value_conv / value_fc1 / value_fc2, weight then bias
enum { CH_ROLE_P1_W = 126, CH_ROLE_P1_B, CH_ROLE_P2_W, CH_ROLE_P2_B, CH_ROLE_V_W, CH_ROLE_V_B, CH_ROLE_F1_W, CH_ROLE_F1_B,
       CH_ROLE_F2_W, CH_ROLE_F2_B, CH_ROLES };

// take(role, entry index, err): called once per role; false stops the resolver with *err set.
using TakeRole = std::function<bool(int, size_t, std::string*)>;
// role_entry[role] = the entry that plays it.  false and *err on a missing tensor, a census or shape mismatch, or a take
// that failed.
bool resolve_net(const std::vector<WeightEntry>& entries, int game, size_t* role_entry /*[NET_ROLES]*/, const TakeRole& take,
                 std::string* err);
bool resolve_chess(const std::vector<WeightEntry>& entries, size_t* role_entry /*[CH_ROLES]*/, const TakeRole& take, std::string* err);

// The per-tensor checks of both paths (no negative dimension, a dtype they read): the size of one element and *count
// elements, or 0 with *err naming the tensor.
size_t element_size(const WeightEntry& t, size_t* count, std::string* err);

}  // namespace spb
