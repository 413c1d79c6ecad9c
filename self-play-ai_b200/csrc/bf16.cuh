// bf16.cuh — the rounding of folded f32 weights to the bf16 operands of the evaluators, shared by the host packers
// (evaluator.cu, evaluator_umma.cu, chess_net.cu) and the device packers of weights_device.cu, so that both write the same
// bytes.
#pragma once
#include <cstdint>
#include <cstring>

namespace spb {

// Round to nearest, ties to even; Inf and NaN are truncated (a NaN whose payload sits in the low 16 bits becomes Inf).
__host__ __device__ inline uint16_t f2bf(float f) {
  uint32_t u;
  std::memcpy(&u, &f, 4);
  if ((u & 0x7F800000u) == 0x7F800000u) return (uint16_t)(u >> 16);
  u += 0x7FFFu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}

}  // namespace spb
