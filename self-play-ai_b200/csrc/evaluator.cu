// evaluator.cu — policy/value evaluation of the gathered leaf batch.
//
// Replaces the tensor part of Model::predict (ref: src/model/mod.rs:60-67,95) and Net::forward
// (ref: src/model/connect_four.rs:75-81; architecture model/mod.rs:152-184, connect_four.rs:50-73):
//   encode (3 planes) -> stem conv3x3+BN+ReLU -> 4 x [conv-BN-ReLU-conv-BN, +skip, ReLU]
//   -> policy head conv3x3(64->32)+BN+ReLU -> Linear -> softmax
//   -> value  head conv3x3(64->3)+BN+ReLU  -> Linear -> tanh
// BatchNorm (eval) is folded into the convs on the host; weights are bf16, accumulation f32,
// activations are rounded to bf16 between layers (both kernels do the same roundings).
//
// Two kernels:
//   k_eval_umma  — the product path: implicit-GEMM 3x3 convs on tcgen05 tensor cores, accumulators
//                  in TMEM, weights streamed by TMA bulk copies (see evaluator_umma.cuh).
//   k_eval_simt  — CUDA-core cross-check of the same arithmetic (SPB_FLAG_EVAL_SIMT), used by tests
//                  to localise a disagreement; never selected implicitly.
#include <cuda_bf16.h>

#include <cstring>
#include <vector>

#include "bf16.cuh"
#include "evaluator.cuh"
#include "evaluator_umma.cuh"

namespace spb {

namespace {

__device__ __forceinline__ float bf16_bits_to_float(uint16_t b) { return __uint_as_float((uint32_t)b << 16); }
__device__ __forceinline__ float round_bf16(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

// 3x3 conv, pad 1, over one board held in shared memory: in[IC][P] -> f(oc, p, acc + bias).
template <class G, class F>
__device__ __forceinline__ void conv3x3_simt(const float* in, int IC, const uint16_t* __restrict__ w, const float* __restrict__ bias,
                                             int OC, F&& f) {
  constexpr int R = G::ROWS, C = G::COLS, P = R * C;
  for (int idx = threadIdx.x; idx < OC * P; idx += blockDim.x) {
    const int oc = idx / P, p = idx % P, r = p / C, c = p % C;
    const uint16_t* wr = w + (size_t)oc * IC * 9;
    float acc = 0.0f;
    for (int ic = 0; ic < IC; ++ic) {
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
        const int rr = r + ky - 1;
        if (rr < 0 || rr >= R) continue;
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const int cc = c + kx - 1;
          if (cc < 0 || cc >= C) continue;
          acc = fmaf(bf16_bits_to_float(wr[ic * 9 + ky * 3 + kx]), in[ic * P + rr * C + cc], acc);
        }
      }
    }
    f(oc, p, acc + bias[oc]);
  }
}

template <class G>
__global__ void __launch_bounds__(256) k_eval_simt(Evaluator::DevNet net, const PState* __restrict__ states,
                                                   const uint32_t* __restrict__ list, const uint32_t* __restrict__ count,
                                                   uint32_t max_n, float* out, int stride, float* logits_out) {
  constexpr int R = G::ROWS, C = G::COLS, P = R * C, A = G::A;
  __shared__ float xa[NET_HIDDEN * P];
  __shared__ float ha[NET_HIDDEN * P];
  __shared__ float head[(NET_POLICY_CH + NET_VALUE_CH) * P];
  __shared__ float logits[A + 1];
  const uint32_t n = min(*count, max_n);
  for (uint32_t i = blockIdx.x; i < n; i += gridDim.x) {
    const uint32_t slot = list ? list[i] : i;
    const PState st = states[slot];
    for (int idx = threadIdx.x; idx < 3 * P; idx += blockDim.x) {
      int plane = idx / P, p = idx % P;
      ha[idx] = G::encode_cell(st, plane, p / C, p % C);                       // get_encoding
    }
    __syncthreads();
    conv3x3_simt<G>(ha, 3, net.w_simt[0], net.bias[0], NET_HIDDEN,
                    [&](int oc, int p, float v) { xa[oc * P + p] = round_bf16(fmaxf(v, 0.0f)); });   // stem
    __syncthreads();
    for (int b = 0; b < NET_BLOCKS; ++b) {                                     // resnet_block, model/mod.rs:152-165
      conv3x3_simt<G>(xa, NET_HIDDEN, net.w_simt[1 + 2 * b], net.bias[1 + 2 * b], NET_HIDDEN,
                      [&](int oc, int p, float v) { ha[oc * P + p] = round_bf16(fmaxf(v, 0.0f)); });
      __syncthreads();
      conv3x3_simt<G>(ha, NET_HIDDEN, net.w_simt[2 + 2 * b], net.bias[2 + 2 * b], NET_HIDDEN,
                      [&](int oc, int p, float v) { xa[oc * P + p] = round_bf16(fmaxf(v + xa[oc * P + p], 0.0f)); });   // (x + f(x)).relu()
      __syncthreads();
    }
    conv3x3_simt<G>(xa, NET_HIDDEN, net.w_simt[9], net.bias[9], NET_POLICY_CH,
                    [&](int oc, int p, float v) { head[oc * P + p] = fmaxf(v, 0.0f); });
    conv3x3_simt<G>(xa, NET_HIDDEN, net.w_simt[10], net.bias[10], NET_VALUE_CH,
                    [&](int oc, int p, float v) { head[(NET_POLICY_CH + oc) * P + p] = fmaxf(v, 0.0f); });
    __syncthreads();
    // Linear layers: one warp per output (flat_view index = channel*P + row*C + col).
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int o = warp; o < A + 1; o += (int)(blockDim.x >> 5)) {
      const bool is_value = o == A;
      const int K = is_value ? NET_VALUE_CH * P : NET_POLICY_CH * P;
      const float* wrow = is_value ? net.vfc_w : net.pfc_w + (size_t)o * K;
      const float* src = is_value ? head + NET_POLICY_CH * P : head;
      float acc = 0.0f;
      for (int k = lane; k < K; k += 32) acc = fmaf(wrow[k], src[k], acc);
#pragma unroll
      for (int off = 16; off >= 1; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
      if (lane == 0) logits[o] = acc + (is_value ? net.vfc_b[0] : net.pfc_b[o]);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      float m = logits[0];
      for (int a = 1; a < A; ++a) m = fmaxf(m, logits[a]);
      float e[A], s = 0.0f;
      for (int a = 0; a < A; ++a) { e[a] = expf(logits[a] - m); s += e[a]; }
      float* o = out + (size_t)slot * stride;
      for (int a = 0; a < A; ++a) o[a] = e[a] / s;                             // softmax, model/mod.rs:63
      o[A] = tanhf(logits[A]);                                                 // connect_four.rs:71
      if (logits_out) for (int a = 0; a < A; ++a) logits_out[(size_t)slot * A + a] = logits[a];
    }
    __syncthreads();
  }
}

}  // namespace

Evaluator::~Evaluator() {
  if (d_blob_) cudaFree(d_blob_);
}

double Evaluator::flops_per_position() const {
  const double P = (double)rows_ * cols_;
  double macs = P * 9.0 * (3.0 * NET_HIDDEN + 2.0 * NET_BLOCKS * NET_HIDDEN * NET_HIDDEN + NET_HIDDEN * (NET_POLICY_CH + NET_VALUE_CH));
  macs += NET_POLICY_CH * P * actions_ + NET_VALUE_CH * P;
  return 2.0 * macs;
}

Evaluator::Layout Evaluator::layout(int game) {
  const bool c4 = game == SPB_GAME_CONNECT4;
  const size_t P = c4 ? 42 : 9, A = c4 ? 7 : 9;
  Layout L;
  // all sections 256-byte aligned; the gaps are zero
  auto reserve = [&](size_t bytes) { const size_t off = (L.bytes + 255) & ~(size_t)255; L.bytes = off + bytes; return off; };
  for (int i = 0; i < NET_CONVS; ++i) {
    const size_t oc = i <= 8 ? NET_HIDDEN : (i == 9 ? NET_POLICY_CH : NET_VALUE_CH), ic = i == 0 ? 3 : NET_HIDDEN;
    L.wsimt[i] = reserve(oc * ic * 9 * 2);
    L.bias[i] = reserve(oc * 4);
  }
  L.pw = reserve(A * NET_POLICY_CH * P * 4);
  L.pb = reserve(A * 4);
  L.vw = reserve(NET_VALUE_CH * P * 4);
  L.vb = reserve(4);
  L.umma = reserve(umma::image_layout(game).bytes);
  return L;
}

void Evaluator::point_at(int game) {
  const Layout L = layout(game);
  const uint8_t* d = static_cast<const uint8_t*>(d_blob_);
  for (int i = 0; i < NET_CONVS; ++i) {
    dev_.w_simt[i] = reinterpret_cast<const uint16_t*>(d + L.wsimt[i]);
    dev_.bias[i] = reinterpret_cast<const float*>(d + L.bias[i]);
  }
  dev_.pfc_w = reinterpret_cast<const float*>(d + L.pw);
  dev_.pfc_b = reinterpret_cast<const float*>(d + L.pb);
  dev_.vfc_w = reinterpret_cast<const float*>(d + L.vw);
  dev_.vfc_b = reinterpret_cast<const float*>(d + L.vb);
  dev_.w_umma = reinterpret_cast<const uint16_t*>(d + L.umma);
  game_ = game;
  rows_ = dev_.rows = game == SPB_GAME_CONNECT4 ? 6 : 3;
  cols_ = dev_.cols = game == SPB_GAME_CONNECT4 ? 7 : 3;
  actions_ = dev_.actions = game == SPB_GAME_CONNECT4 ? 7 : 9;
}

bool Evaluator::upload(const HostNet& net, std::string* err) {
  const Layout L = layout(net.game);
  std::vector<uint8_t> blob(L.bytes, 0);
  for (int i = 0; i < NET_CONVS; ++i) {
    const auto& c = net.conv[i];
    uint16_t* w = reinterpret_cast<uint16_t*>(blob.data() + L.wsimt[i]);
    for (size_t k = 0; k < c.w.size(); ++k) w[k] = f2bf(c.w[k]);
    std::memcpy(blob.data() + L.bias[i], c.b.data(), (size_t)c.oc * 4);
  }
  std::memcpy(blob.data() + L.pw, net.pfc_w.data(), net.pfc_w.size() * 4);
  std::memcpy(blob.data() + L.pb, net.pfc_b.data(), net.pfc_b.size() * 4);
  std::memcpy(blob.data() + L.vw, net.vfc_w.data(), net.vfc_w.size() * 4);
  std::memcpy(blob.data() + L.vb, net.vfc_b.data(), net.vfc_b.size() * 4);
  // tcgen05 operand images + epilogue tables
  std::vector<uint8_t> umma_img;
  umma::pack_weights(net, &umma_img);
  std::memcpy(blob.data() + L.umma, umma_img.data(), umma_img.size());

  // new image first, then swap: a failed upload keeps the previous checkpoint usable
  void* nblob = nullptr;
  cudaError_t e = cudaMalloc(&nblob, blob.size());
  if (e == cudaSuccess) e = cudaMemcpy(nblob, blob.data(), blob.size(), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    if (nblob) cudaFree(nblob);
    cudaGetLastError();
    *err = std::string("weight upload: ") + cudaGetErrorString(e);
    return false;
  }
  if (d_blob_) cudaFree(d_blob_);
  d_blob_ = nblob;
  blob_bytes_ = blob.size();
  point_at(net.game);
  loaded_ = true;
  return true;
}

uint8_t* Evaluator::image_for(int game, std::string* err) {
  const size_t bytes = layout(game).bytes;
  if (!d_blob_ || blob_bytes_ != bytes) {
    void* nblob = nullptr;
    const cudaError_t e = cudaMalloc(&nblob, bytes);
    if (e != cudaSuccess) {
      cudaGetLastError();
      *err = std::string("weight image: ") + cudaGetErrorString(e);
      return nullptr;
    }
    if (d_blob_) cudaFree(d_blob_);
    d_blob_ = nblob;
    blob_bytes_ = bytes;
    loaded_ = false;
    point_at(game);
  }
  return static_cast<uint8_t*>(d_blob_);
}

cudaError_t Evaluator::launch(const PState* states, const uint32_t* list, const uint32_t* count_dev, uint32_t max_n, float* out,
                              int stride, float* logits_out, bool simt, cudaStream_t stream, bool overlap) {
  if (!loaded_) return cudaErrorNotReady;
  if (simt) {
    const unsigned grid = std::min<unsigned>(max_n, 148u * 4u);
    if (game_ == SPB_GAME_CONNECT4)
      k_eval_simt<Connect4><<<grid, 256, 0, stream>>>(dev_, states, list, count_dev, max_n, out, stride, logits_out);
    else
      k_eval_simt<TicTacToe><<<grid, 256, 0, stream>>>(dev_, states, list, count_dev, max_n, out, stride, logits_out);
    return cudaGetLastError();
  }
  return umma::launch(dev_, game_, states, list, count_dev, max_n, out, stride, logits_out, stream, overlap);
}

cudaError_t Evaluator::launch_ring(const Trees& T, const AsyncCtl& C, cudaStream_t stream) {
  if (!loaded_) return cudaErrorNotReady;
  return umma::launch_ring(dev_, game_, T, C, stream);
}

}  // namespace spb
