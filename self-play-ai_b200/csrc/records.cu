// records.cu — trajectory records on the device (declarations and contracts in records.cuh).
//
// Ordering.  An output buffer holds whole trajectories as contiguous runs in ply order (reserve_output reserves a game's
// records at once; emit_and_finish / emit_game write them), and a gathered buffer is a concatenation of such buffers.
// So the (game id, ply) order is a permutation of runs: find the run heads (a new game id, or a break in consecutive
// plies), sort the runs by (game id, first ply) with two stable radix sorts (first ply, then game id), scan the sorted
// lengths into destination offsets, and move every record once.  With unique (game id, ply) keys the runs of one game
// cover disjoint ply intervals, so this is exactly the order of record_order (trajectory.cuh).  The sort works on one key
// per run (a few per game), the move on every byte: the move is the bandwidth-bound kernel, flat over 8-byte words, so a
// 512-ply chess run (830 KB) costs the same per byte as a 7-ply Connect4 one.
//
// Training tensors.  Rows of 126 / 27 encoding floats and 7 / 9 policy floats are not 16-byte multiples, so each output
// is written as one flat array: consecutive lanes write consecutive floats, 16-byte streaming stores from the first
// 16-byte boundary of the array, scalar stores before it and after the last whole float4; every float is written once.
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "host_engine.hpp"
#include "records.cuh"

namespace spb {
namespace {

constexpr int THREADS = 256;

template <class Rec>
struct IsRunHead {
  const Rec* src;
  const unsigned long long* ids;
  __device__ __forceinline__ bool operator()(uint32_t i) const {
    return i == 0 || ids[i] != ids[i - 1] || (uint32_t)src[i].ply != (uint32_t)src[i - 1].ply + 1u;
  }
};

template <class Rec>
__global__ void __launch_bounds__(THREADS) k_run_first_ply(const Rec* __restrict__ src, const uint32_t* __restrict__ run_start, uint32_t m,
                                                           uint32_t* __restrict__ ply_key, uint32_t* __restrict__ run) {
  for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < m; r += gridDim.x * blockDim.x) {
    ply_key[r] = src[run_start[r]].ply;
    run[r] = r;
  }
}

__global__ void __launch_bounds__(THREADS) k_run_game_id(const unsigned long long* __restrict__ ids, const uint32_t* __restrict__ run_start,
                                                         const uint32_t* __restrict__ run, uint32_t m, unsigned long long* __restrict__ id_key) {
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < m; j += gridDim.x * blockDim.x) id_key[j] = ids[run_start[run[j]]];
}

// len[j]: records of the j-th run in (game id, first ply) order
__global__ void __launch_bounds__(THREADS) k_run_length(const uint32_t* __restrict__ run_start, const uint32_t* __restrict__ order, uint32_t m,
                                                        uint32_t n, uint32_t* __restrict__ len) {
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < m; j += gridDim.x * blockDim.x) {
    const uint32_t r = order[j];
    len[j] = (r + 1 < m ? run_start[r + 1] : n) - run_start[r];
  }
}

// src_of[destination record] = source record; one warp per sorted run, its lanes on consecutive records
__global__ void __launch_bounds__(THREADS) k_source_map(const uint32_t* __restrict__ run_start, const uint32_t* __restrict__ order,
                                                        const uint32_t* __restrict__ off, const uint32_t* __restrict__ len, uint32_t m,
                                                        uint32_t* __restrict__ src_of) {
  const uint32_t lane = threadIdx.x & 31, warps = gridDim.x * (blockDim.x / 32);
  for (uint32_t j = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32; j < m; j += warps) {
    const uint32_t s = run_start[order[j]], d = off[j], l = len[j];
    for (uint32_t k = lane; k < l; k += 32) src_of[d + k] = s + k;
  }
}

// dst[k] = src[src_of[k]], flat over the 8-byte words of the destination: consecutive lanes read and write consecutive
// words of a record, UNROLL independent loads in flight per thread.  Streaming loads and stores: neither side is read
// again by this call.
template <class Rec>
__global__ void __launch_bounds__(THREADS) k_move_records(const Rec* __restrict__ src, const unsigned long long* __restrict__ src_ids,
                                                          const uint32_t* __restrict__ src_of, uint32_t n, Rec* __restrict__ dst,
                                                          unsigned long long* __restrict__ dst_ids) {
  constexpr uint32_t W = sizeof(Rec) / 8;
  constexpr int UNROLL = 4;
  const auto* s = reinterpret_cast<const unsigned long long*>(src);
  auto* d = reinterpret_cast<unsigned long long*>(dst);
  const unsigned long long total = (unsigned long long)n * W, stride = (unsigned long long)gridDim.x * blockDim.x;
  const unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  for (unsigned long long w0 = t; w0 < total; w0 += stride * UNROLL) {
    unsigned long long v[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const unsigned long long w = w0 + u * stride;
      if (w < total) {
        const uint32_t k = (uint32_t)(w / W), j = (uint32_t)(w - (unsigned long long)k * W);
        v[u] = __ldcs(s + (unsigned long long)__ldg(src_of + k) * W + j);
      }
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const unsigned long long w = w0 + u * stride;
      if (w < total) __stcs(d + w, v[u]);
    }
  }
  if (dst_ids)
    for (unsigned long long k = t; k < n; k += stride) __stcs(dst_ids + k, __ldcs(src_ids + __ldg(src_of + k)));
}

// Byte offsets of order_records' arrays in its scratch, for n records and cub_bytes of CUB temporaries.
struct OrderScratch {
  size_t run_start, n_runs, key_a[2], run[2], id_key[2], src_of, cub, bytes;
  OrderScratch(size_t n, size_t cub_bytes) {
    StageLayout L;
    run_start = L.take(n * 4);
    n_runs = L.take(4);
    for (int b = 0; b < 2; ++b) key_a[b] = L.take(n * 4);       // first plies; reused for the run lengths and offsets
    for (int b = 0; b < 2; ++b) run[b] = L.take(n * 4);
    for (int b = 0; b < 2; ++b) id_key[b] = L.take(n * 8);
    src_of = L.take(n * 4);
    cub = L.take(cub_bytes);
    bytes = L.bytes;
  }
};

// Bytes of CUB temporaries for the select over n records and the sorts and scan over up to n runs.
template <class Rec>
size_t cub_bytes(uint32_t n) {
  const uint32_t m = n;
  size_t need = 0, b = 0;
  cub::DeviceSelect::If(nullptr, b, thrust::counting_iterator<uint32_t>(0), (uint32_t*)nullptr, (uint32_t*)nullptr, (int)n,
                        IsRunHead<Rec>{nullptr, nullptr});
  need = std::max(need, b);
  cub::DoubleBuffer<uint32_t> k32, v32;
  cub::DoubleBuffer<unsigned long long> k64;
  cub::DeviceRadixSort::SortPairs(nullptr, b, k32, v32, (int)m, 0, (int)sizeof(Rec::ply) * 8);
  need = std::max(need, b);
  cub::DeviceRadixSort::SortPairs(nullptr, b, k64, v32, (int)m);
  need = std::max(need, b);
  cub::DeviceScan::ExclusiveSum(nullptr, b, (uint32_t*)nullptr, (uint32_t*)nullptr, (int)m);
  return std::max(need, b);
}

unsigned grid_for(size_t items, int per_block) {
  return (unsigned)std::max<size_t>(1, std::min<size_t>((items + per_block - 1) / per_block, (size_t)1 << 16));
}

template <class Shape>
__global__ void __launch_bounds__(THREADS) k_training(const spb_position* __restrict__ pos, const unsigned long long* __restrict__ indices,
                                                      unsigned long long n, float* encodings, float* policies, float* values) {
  constexpr int R = Shape::R, C = Shape::C, A = Shape::A, E = 3 * R * C;
  const int part = blockIdx.y;                                         // 0 encodings, 1 policies, 2 values
  float* out = part == 0 ? encodings : part == 1 ? policies : values;
  if (!out) return;
  const unsigned long long total = n * (unsigned long long)(part == 0 ? E : part == 1 ? A : 1);
  const auto value = [&](unsigned long long f) -> float {
    if (part == 0) {
      const unsigned long long row = f / E;
      const int cell = (int)(f - row * E), plane = cell / (R * C), r = (cell % (R * C)) / C, c = cell % C;
      const spb_position& p = pos[indices ? __ldg(indices + row) : row];
      const int cp = __ldg(&p.current_player) & 1;                   // as the host reads it: the low bit only
      const int bit = Shape::bit(r, c);
      const uint32_t m = (uint32_t)(__ldg(&p.stones[cp]) >> bit) & 1u, q = (uint32_t)(__ldg(&p.stones[cp ^ 1]) >> bit) & 1u;
      return plane == 0 ? (m ? 1.0f : 0.0f) : plane == 1 ? (q ? 1.0f : 0.0f) : ((m | q) ? 0.0f : 1.0f);
    }
    if (part == 1) {
      const unsigned long long row = f / A;
      const int a = (int)(f - row * A);
      const spb_position& p = pos[indices ? __ldg(indices + row) : row];
      float s = 0.0f;
#pragma unroll
      for (int b = 0; b < A; ++b) s += (float)__ldg(&p.visit_counts[b]);   // the host's f32 sum, in the same order
      return (float)__ldg(&p.visit_counts[a]) / s;                         // IEEE divide (no fast-math in this build)
    }
    return (float)__ldg(&pos[indices ? __ldg(indices + f) : f].outcome);
  };
  // floats before the first 16-byte boundary, whole float4s, then the tail
  const unsigned long long lead = ((16u - (reinterpret_cast<uintptr_t>(out) & 15u)) & 15u) / 4u, head = lead < total ? lead : total;
  const unsigned long long body = (total - head) / 4, tail0 = head + 4 * body;
  const unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x, stride = (unsigned long long)gridDim.x * blockDim.x;
  for (unsigned long long q = t; q < body; q += stride) {
    const unsigned long long f = head + 4 * q;
    __stcs(reinterpret_cast<float4*>(out + f), make_float4(value(f), value(f + 1), value(f + 2), value(f + 3)));
  }
  for (unsigned long long e = t; e < head + (total - tail0); e += stride) {
    const unsigned long long f = e < head ? e : tail0 + (e - head);
    out[f] = value(f);
  }
}

struct Connect4Shape {
  static constexpr int R = 6, C = 7, A = 7;
  __device__ static int bit(int r, int c) { return c * 7 + r; }
};
struct TicTacToeShape {
  static constexpr int R = 3, C = 3, A = 9;
  __device__ static int bit(int r, int c) { return r * 3 + c; }
};

__global__ void __launch_bounds__(THREADS) k_index_check(const unsigned long long* __restrict__ indices, unsigned long long n,
                                                         unsigned long long n_positions, unsigned long long* bad) {
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x)
    if (indices[i] >= n_positions) atomicMin(bad, i);
}

}  // namespace

template <class Rec>
size_t order_scratch_bytes(size_t n) {
  return OrderScratch(n, cub_bytes<Rec>((uint32_t)n)).bytes;
}

template <class Rec>
cudaError_t order_records(const Rec* src, const unsigned long long* src_ids, size_t n_, Rec* dst, unsigned long long* dst_ids,
                          void* scratch, cudaStream_t stream) {
  if (n_ == 0) return cudaSuccess;
  if (n_ >= ((size_t)1 << 31)) return cudaErrorInvalidValue;
  const uint32_t n = (uint32_t)n_;
  const OrderScratch S(n, cub_bytes<Rec>(n));
  char* base = static_cast<char*>(scratch);
  const auto at = [base](size_t off) { return reinterpret_cast<uint32_t*>(base + off); };
  uint32_t* run_start = at(S.run_start);
  uint32_t* d_runs = at(S.n_runs);
  void* tmp = base + S.cub;
  size_t tmp_bytes = S.bytes - S.cub;
  cudaError_t ce = cub::DeviceSelect::If(tmp, tmp_bytes, thrust::counting_iterator<uint32_t>(0), run_start, d_runs, (int)n,
                                         IsRunHead<Rec>{src, src_ids}, stream);
  uint32_t m = 0;
  if (ce == cudaSuccess) ce = cudaMemcpyAsync(&m, d_runs, 4, cudaMemcpyDeviceToHost, stream);
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(stream);
  if (ce != cudaSuccess) return ce;
  // runs by first ply, then (stable) by game id
  cub::DoubleBuffer<uint32_t> ply(at(S.key_a[0]), at(S.key_a[1])), run(at(S.run[0]), at(S.run[1]));
  cub::DoubleBuffer<unsigned long long> id(reinterpret_cast<unsigned long long*>(base + S.id_key[0]),
                                           reinterpret_cast<unsigned long long*>(base + S.id_key[1]));
  k_run_first_ply<Rec><<<grid_for(m, THREADS), THREADS, 0, stream>>>(src, run_start, m, ply.Current(), run.Current());
  tmp_bytes = S.bytes - S.cub;
  ce = cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, ply, run, (int)m, 0, (int)sizeof(Rec::ply) * 8, stream);
  if (ce != cudaSuccess) return ce;
  k_run_game_id<<<grid_for(m, THREADS), THREADS, 0, stream>>>(src_ids, run_start, run.Current(), m, id.Current());
  tmp_bytes = S.bytes - S.cub;
  ce = cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, id, run, (int)m, 0, 64, stream);
  if (ce != cudaSuccess) return ce;
  // lengths in run order, their exclusive scan = destination offsets
  uint32_t* len = at(S.key_a[0]);
  uint32_t* off = at(S.key_a[1]);
  k_run_length<<<grid_for(m, THREADS), THREADS, 0, stream>>>(run_start, run.Current(), m, n, len);
  tmp_bytes = S.bytes - S.cub;
  ce = cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, len, off, (int)m, stream);
  if (ce != cudaSuccess) return ce;
  uint32_t* src_of = at(S.src_of);
  k_source_map<<<grid_for(m, THREADS / 32), THREADS, 0, stream>>>(run_start, run.Current(), off, len, m, src_of);
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const size_t words = (size_t)n * (sizeof(Rec) / 8);
  k_move_records<Rec><<<(unsigned)std::min<size_t>(grid_for(words, THREADS), (size_t)sms * 8), THREADS, 0, stream>>>(src, src_ids, src_of,
                                                                                                                   n, dst, dst_ids);
  return cudaGetLastError();
}

template size_t order_scratch_bytes<spb_position>(size_t);
template size_t order_scratch_bytes<spb_chess_position>(size_t);
template cudaError_t order_records<spb_position>(const spb_position*, const unsigned long long*, size_t, spb_position*,
                                                 unsigned long long*, void*, cudaStream_t);
template cudaError_t order_records<spb_chess_position>(const spb_chess_position*, const unsigned long long*, size_t, spb_chess_position*,
                                                       unsigned long long*, void*, cudaStream_t);

cudaError_t launch_training_tensors(int32_t game, const spb_position* pos, const unsigned long long* indices, size_t n,
                                    float* encodings, float* policies, float* values, int sms, cudaStream_t stream) {
  const int E = game == SPB_GAME_CONNECT4 ? 126 : 27;
  const dim3 grid(std::min<unsigned>(grid_for(n * E / 4 + 1, THREADS), (unsigned)sms * 8), 3);
  if (game == SPB_GAME_CONNECT4)
    k_training<Connect4Shape><<<grid, THREADS, 0, stream>>>(pos, indices, n, encodings, policies, values);
  else
    k_training<TicTacToeShape><<<grid, THREADS, 0, stream>>>(pos, indices, n, encodings, policies, values);
  return cudaGetLastError();
}

cudaError_t launch_index_check(const unsigned long long* indices, size_t n, size_t n_positions, unsigned long long* bad, int sms,
                               cudaStream_t stream) {
  k_index_check<<<std::min<unsigned>(grid_for(n, THREADS), (unsigned)sms * 4), THREADS, 0, stream>>>(indices, n, n_positions, bad);
  return cudaGetLastError();
}

}  // namespace spb
