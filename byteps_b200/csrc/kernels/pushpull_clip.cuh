// Global-norm gradient clipping inside the fused optimizer exchange (sm_100a).
//
// The fused kernels of pushpull.cu update the weights in the same launch that reduces the gradients, so there is no
// point at which the averaged gradients exist as a whole.  With clipping the exchange is split in three stream-ordered
// phases that need no host synchronisation (the step still captures into one CUDA graph):
//   1. per bucket: reduce-scatter my shard, scale by 1/world, write it (wire dtype) into my own window and add the
//      squares of the values as written, times grad_scale^2, into fixed per-(bucket, CTA) fp64 slots;
//   2. once per step: sum my slots in a fixed order, publish the sum in the symmetric arena, flag-barrier and add
//      every rank's sum in rank order, so every rank holds a bit-identical norm and clip coefficient;
//   3. per (dtype, optimizer) class: read the averaged shard from local memory, run the SGD/Adam epilogue with
//      scale = coef on the fp32 master/moment shards (streamed through shared memory with bulk copies) and write the
//      new parameters to every replica.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "kernels/pushpull.cuh"

namespace bps {

// One bucket of phase 3.  Offsets are bytes into the arena; master/state are this rank's fp32 shards.
struct ClipDesc {
  uint64_t grad_off;
  uint64_t param_off;
  uint64_t nelem;        // padded element count of the bucket (multiple of 8)
  float* master;
  float* state0;
  float* state1;
  const OptHParams* hp;
  uint64_t pad;
};

// Local device block: max_norm is written by the host with the hyper-parameters, the rest by phase 2.
struct ClipState {
  float max_norm;
  float norm;      // total L2 norm of the averaged, unscaled gradients of the last step (before clipping)
  float coef;      // min(max_norm / (norm + 1e-6), 1); NaN propagates
  uint32_t step;   // completed phase-2 launches: its parity selects the half of the publish region
};

constexpr int kClipSlotsPerBucket = kMaxBlocks;   // phase-1 partial sums, one per CTA
constexpr size_t kClipPublishBytes = 16;          // two fp64 sums (step parity) per rank in the arena

// Phase 1.  slots: this bucket's kClipSlotsPerBucket fp64 entries (entry i written by CTA i; unused entries must
// stay zero).  hp: the bucket's hyper-parameters (grad_scale).
cudaError_t launch_clip_reduce_sumsq(const PeerView& pv, int wire, size_t off_bytes, size_t nelem, float scale,
                                     double* slots, const OptHParams* hp, const LaunchCfg& cfg, cudaStream_t stream);

// Phase 2.  One CTA.  publish_off: kClipPublishBytes in every rank's arena.
cudaError_t launch_clip_finalize(const PeerView& pv, const double* slots, int nslots, size_t publish_off,
                                 ClipState* state, int channel, cudaStream_t stream);

// Phase 3.  descs: device table of ndescs buckets, all of dtype `wire` (gradient == parameter dtype).
cudaError_t launch_clip_update(const PeerView& pv, int wire, int opt_kind, const ClipDesc* descs, int ndescs,
                               const ClipState* state, int blocks, int stages, int use_nvls, int channel,
                               cudaStream_t stream);

}  // namespace bps
