// det.cuh -- the fixed-order gradient sums of the deterministic update (cacto_*_grad_det, include/cacto_b200.h).
//
// A gradient kernel instantiated with DET = true adds its CTA's contribution into slice blockIdx.x of a caller-owned partials
// workspace instead of into the gradient block with atomics (mlp.cuh grad_add).  A slice has the layout of the gradient block
// (n floats) followed by one loss partial, padded to 16 bytes.  The CTAs of a launch are bounded by CACTO_DET_MAX_SLICES: a batch
// of more tiles runs as several launches ("waves") of at most that many CTAs, CTA j of every wave adding into slice j, so the
// slices are written in wave order and stay bounded whatever the batch size.  det_reduce then sums the slices into the
// gradient block in slice order, starting from 0.0f, and adds the result to what the block held.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "cacto_b200.h"

namespace cacto {

__host__ __device__ __forceinline__ int64_t det_stride(int64_t n) { return (n + 1 + 3) & ~(int64_t)3; }
// samples per CTA of the width-generic actor gradient (csrc/actor_width.cu): 4-sample tiles while they fill at most one wave of
// the 148 SMs (latency of the reference's batch sizes), 16-sample tiles beyond
static inline int actor_width_tile(int64_t B) { return B <= 4 * 148 ? 4 : 16; }
// floats of a slice of the tcgen05 engine's partials (update_tc.cu: TC_DET_SLICE)
constexpr int64_t det_tc_slice = 648;
static inline int64_t det_slices(int64_t tiles) { return tiles < CACTO_DET_MAX_SLICES ? tiles : CACTO_DET_MAX_SLICES; }

// grad[i] += sum_j part[j * stride + i] (j = 0 .. slices-1) for i < n; loss[0] += the same sum of the loss partials at i = n
// (loss may be NULL).  Enqueued with programmatic serialization behind the last wave.
int det_reduce(const float* part, int64_t slices, int64_t n, float* grad, float* loss, cudaStream_t st);

}  // namespace cacto
