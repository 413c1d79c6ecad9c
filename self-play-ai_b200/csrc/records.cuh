// records.cuh — trajectory records on the device (records.cu): the (game id, ply) ordering of an output buffer (or of a
// gathered concatenation of them) straight into a caller's device buffer, and the Connect4 / tic-tac-toe training
// tensors of records held in device memory.  Both engines use it (HostEngine::drain_trajectories_device, gather.cu).
#pragma once
#include <cstddef>

#include <cuda_runtime.h>

#include "../../include/selfplay_b200.h"

namespace spb {

// Device scratch bytes order_records needs for n records (run keys, offsets, sort temporaries).
template <class Rec> size_t order_scratch_bytes(size_t n);

// Writes the n records of src / src_ids to dst / dst_ids (nullable) in the order record_order (trajectory.cuh) gives,
// for any buffer whose (game id, ply) keys are unique.  Works on runs — maximal stretches of one game id with
// consecutive plies, which is how reserve_output lays whole trajectories down — sorted by (game id, first ply); every
// record is then moved once.  scratch: order_scratch_bytes(n) device bytes, 16-byte aligned.  Enqueued on `stream`; it
// synchronises once (the run count sizes the sort) and returns before the move has finished.  n < 2^31.
template <class Rec>
cudaError_t order_records(const Rec* src, const unsigned long long* src_ids, size_t n, Rec* dst, unsigned long long* dst_ids,
                          void* scratch, cudaStream_t stream);

// The tensors of spb_positions_to_training(game, ...) for n rows, row i built from pos[indices ? indices[i] : i] (every
// index already checked < n_positions); each output nullable.  Enqueued on `stream`.
cudaError_t launch_training_tensors(int32_t game, const spb_position* pos, const unsigned long long* indices, size_t n,
                                    float* encodings, float* policies, float* values, int sms, cudaStream_t stream);

// bad[0] = the first i < n with indices[i] >= n_positions (atomicMin; the caller sets it to ~0 first).
cudaError_t launch_index_check(const unsigned long long* indices, size_t n, size_t n_positions, unsigned long long* bad, int sms,
                               cudaStream_t stream);

}  // namespace spb
