// evaluator_umma.cuh — interface of the tcgen05 evaluator kernel (evaluator_umma.cu).
#pragma once
#include <cstdint>
#include <vector>

#include "async.cuh"
#include "evaluator.cuh"

namespace spb {
namespace umma {
// Packs the folded net into the device image the kernel streams with cp.async.bulk (UMMA operand layout: kx-triple blocks per kernel row, one block per tap for the stem).
void pack_weights(const HostNet& net, std::vector<uint8_t>* out);
// Where pack_weights puts things, for the device packer (weights_device.cu): the conv layers (stem, 8 residual, fused
// head conv) with their output width N and K chunks of 8 channels, the bias table, the policy / value Linear tables.
struct ImageLayout {
  size_t layer_offset[10];
  int layer_n[10], layer_kchunks[10];
  size_t off_bias, off_wp, off_wv, off_fcb, bytes;
};
ImageLayout image_layout(int game);
// Static work list (spb_predict, lock-step pipeline).  overlap: programmatic dependent launch (set-up may run under the
// previous kernel of the stream).
cudaError_t launch(const Evaluator::DevNet& net, int game, const PState* states, const uint32_t* list,
                   const uint32_t* count_dev, uint32_t max_n, float* out, int stride, float* logits_out,
                   cudaStream_t stream, bool overlap);
// Asynchronous search pipeline: evaluator + tree warps resident until every tree of the search is done (async.cuh).
cudaError_t launch_ring(const Evaluator::DevNet& net, int game, const Trees& T, const AsyncCtl& C, cudaStream_t stream);
}  // namespace umma
}  // namespace spb
