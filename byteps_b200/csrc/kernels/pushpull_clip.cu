// Global-norm gradient clipping kernels (see pushpull_clip.cuh for the three phases).
#include "kernels/pushpull_clip.cuh"

#include "kernels/common.cuh"
#include "kernels/pushpull_dev.cuh"

namespace bps {

namespace {

// Sum of v over the CTA in a fixed order (shuffle tree per warp, warps in index order); valid in thread 0.
// blockDim.x must be a multiple of 32.
__device__ __forceinline__ double block_sum_f64(double v) {
  __shared__ double warp_sums[32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += warp_sums[w];
  return t;
}

// ---------------------------------------------------------------- phase 1
// No closing barrier: peers may still read my window when this CTA exits, but nothing writes the gradient windows
// before phase 2, whose barrier every rank reaches only after all of its phase-1 launches.
template <class W>
__global__ void __launch_bounds__(512) clip_reduce_sumsq_kernel(PeerView pv, size_t off, size_t total_groups,
                                                                float scale, double* slots, const OptHParams* hp,
                                                                int nvls, int channel) {
  constexpr int E = W::kPerVec;
  size_t s0, s1;
  shard_units_of<E>(total_groups, pv.world, pv.rank, &s0, &s1);
  barrier_peers(pv, channel);
  char* mine = pv.data[pv.rank] + off;
  EpiScale epi{scale};
  double ss = 0.0;
  reduce_phase<W, kUnroll>(pv, off, s0, s1, nvls != 0, rot_of(pv), epi, [&](const float* f, size_t unit) {
    const Vec16 v = W::pack(f);
    st_stream16(mine + unit * 16, v);
    float w[E];
    W::unpack(v, w);     // the norm is of the values as written (wire dtype)
#pragma unroll
    for (int k = 0; k < E; ++k) ss += (double)w[k] * (double)w[k];
  });
  ss = block_sum_f64(ss);
  if (threadIdx.x == 0) {
    const double gs = (double)hp->grad_scale;
    slots[blockIdx.x] = ss * gs * gs;
  }
}

// ---------------------------------------------------------------- phase 2
__global__ void __launch_bounds__(256) clip_finalize_kernel(PeerView pv, const double* slots, int nslots,
                                                            size_t pub_off, ClipState* st, int channel) {
  double v = 0.0;
  for (int i = threadIdx.x; i < nslots; i += blockDim.x) v += slots[i];
  v = block_sum_f64(v);
  // Two halves by step parity: a rank that runs ahead into the next step writes the other half, and it cannot get
  // two steps ahead because this step's barrier (and phase 3's) needs every peer.
  const uint32_t parity = st->step & 1u;
  if (threadIdx.x == 0) reinterpret_cast<volatile double*>(pv.data[pv.rank] + pub_off)[parity] = v;
  barrier_peers(pv, channel);
  if (threadIdx.x == 0) {
    double tot = 0.0;
    for (int p = 0; p < pv.world; ++p) tot += reinterpret_cast<const volatile double*>(pv.data[p] + pub_off)[parity];
    const float norm = (float)sqrt(tot);
    float coef = st->max_norm / (norm + 1e-6f);
    if (coef > 1.f) coef = 1.f;   // clamp that keeps NaN (fminf(nan, 1) would return 1)
    st->norm = norm;
    st->coef = coef;
    st->step += 1u;
  }
}

// ---------------------------------------------------------------- phase 3
// Same shared-memory ring as pushpull_fused_opt_tma_kernel (pushpull.cu): a producer warp bulk-copies the fp32 state
// tiles, the consumers update them in place and one thread writes them back.  The tiles of all descriptors form one
// sequence dealt round-robin to the CTAs, so small buckets do not leave CTAs idle.
constexpr int kClipTileUnits = 256;
constexpr int kClipThreads = kClipTileUnits + 32;
constexpr int kClipMaxStages = 8;

struct ClipSmem {
  uint64_t full[kClipMaxStages];
  uint64_t empty[kClipMaxStages];
};

__device__ __forceinline__ void make_epi(EpiSGD& e, const ClipDesc& d, size_t shard_begin, float coef) {
  e = EpiSGD{d.master, d.state0, shard_begin, coef, *d.hp};
}
__device__ __forceinline__ void make_epi(EpiAdam& e, const ClipDesc& d, size_t shard_begin, float coef) {
  e = EpiAdam{d.master, d.state0, d.state1, shard_begin, coef, *d.hp};
}

// on_desc(d, s0) before the first tile of descriptor d this CTA owns; on_tile(d, s0, t, units) for each of them.
// Producer and consumers walk the identical sequence.
template <int E, class D, class T>
__device__ __forceinline__ void for_clip_tiles(const PeerView& pv, const ClipDesc* descs, int ndescs, D&& on_desc,
                                               T&& on_tile) {
  size_t before = 0;   // tiles of the earlier descriptors
  for (int d = 0; d < ndescs; ++d) {
    size_t s0, s1;
    shard_units_of<E>(descs[d].nelem / 8, pv.world, pv.rank, &s0, &s1);
    const size_t ntiles = (s1 - s0 + kClipTileUnits - 1) / kClipTileUnits;
    size_t k = (blockIdx.x + gridDim.x - before % gridDim.x) % gridDim.x;
    if (k < ntiles) on_desc(d, s0);
    for (; k < ntiles; k += gridDim.x) {
      const size_t t = s0 + k * kClipTileUnits;
      const size_t left = s1 - t;
      on_tile(d, s0, t, (uint32_t)(left < (size_t)kClipTileUnits ? left : (size_t)kClipTileUnits));
    }
    before += ntiles;
  }
}

template <int E>
__device__ __forceinline__ void lds_f(const unsigned char* p, float* f) {
#pragma unroll
  for (int k = 0; k < E; k += 4) {
    Vec16 v = lds16(p + k * 4);
    f[k] = __uint_as_float(v.x); f[k + 1] = __uint_as_float(v.y);
    f[k + 2] = __uint_as_float(v.z); f[k + 3] = __uint_as_float(v.w);
  }
}
template <int E>
__device__ __forceinline__ void sts_f(unsigned char* p, const float* f) {
#pragma unroll
  for (int k = 0; k < E; k += 4)
    sts16(p + k * 4, Vec16{__float_as_uint(f[k]), __float_as_uint(f[k + 1]), __float_as_uint(f[k + 2]),
                           __float_as_uint(f[k + 3])});
}

template <class W, class Epi>
__global__ void __launch_bounds__(kClipThreads, 2) clip_update_kernel(PeerView pv, const ClipDesc* descs, int ndescs,
                                                                      const ClipState* st, int nvls, int stages,
                                                                      int channel) {
  constexpr int E = W::kPerVec;
  constexpr uint32_t kUnitBytes = E * 4;
  constexpr size_t kStreamBytes = (size_t)kClipTileUnits * kUnitBytes;
  constexpr size_t kStageBytes = Epi::kStreams * kStreamBytes;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  ClipSmem* sm = reinterpret_cast<ClipSmem*>(smem_raw);
  unsigned char* ring = smem_raw + 128;   // [stage][stream][kStreamBytes]
  const float coef = st->coef;
  const bool is_producer = (threadIdx.x >> 5) == (kClipTileUnits >> 5);
  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(&sm->full[s], 1);
      mbar_init(&sm->empty[s], 1);
    }
    mbar_fence_init();
  }
  __syncthreads();

  Epi epi;
  int s = 0;
  uint32_t phase = 0;
  if (is_producer) {
    if ((threadIdx.x & 31) == 0) {
      int nstreams = 0;
      for_clip_tiles<E>(
          pv, descs, ndescs,
          [&](int d, size_t s0) {
            make_epi(epi, descs[d], s0 * E, coef);
            nstreams = epi.active_streams();
          },
          [&](int, size_t s0, size_t t, uint32_t units) {
            const uint32_t bytes = units * kUnitBytes;
            mbar_wait(&sm->empty[s], phase ^ 1);   // slot written back (first pass falls through)
            mbar_arrive_expect_tx(&sm->full[s], bytes * nstreams);
            unsigned char* dst = ring + (size_t)s * kStageBytes;
            const size_t li = (t - s0) * E;
            for (int i = 0; i < nstreams; ++i)
              bulk_g2s(dst + (size_t)i * kStreamBytes, epi.stream(i) + li, bytes, &sm->full[s]);
            if (++s == stages) {
              s = 0;
              phase ^= 1;
            }
          });
    }
  } else {
    const char* mine = pv.data[pv.rank];
    int prev_s = -1, nstreams = 0;
    for_clip_tiles<E>(
        pv, descs, ndescs,
        [&](int d, size_t s0) {
          make_epi(epi, descs[d], s0 * E, coef);
          nstreams = epi.active_streams();
        },
        [&](int d, size_t s0, size_t t, uint32_t units) {
          const size_t unit = t + threadIdx.x;
          const bool valid = threadIdx.x < units;
          // the averaged gradient phase 1 left in my own window (local HBM), requested before the state wait
          Vec16 g{0u, 0u, 0u, 0u};
          if (valid) g = ld_stream16(mine + descs[d].grad_off + unit * 16);
          unsigned char* slot = ring + (size_t)s * kStageBytes;
          mbar_wait(&sm->full[s], phase);
          if (valid) {
            float acc[E];
            W::unpack(g, acc);
            typename Epi::template State<E> stt;
            for (int i = 0; i < nstreams; ++i)
              lds_f<E>(slot + (size_t)i * kStreamBytes + threadIdx.x * kUnitBytes, epi.template field<E>(stt, i));
            epi.template update<E>(acc, stt);
            for (int i = 0; i < nstreams; ++i)
              sts_f<E>(slot + (size_t)i * kStreamBytes + threadIdx.x * kUnitBytes, epi.template field<E>(stt, i));
            sink_peers<W, E>(pv, descs[d].param_off, unit, acc, nvls != 0);   // new parameters to every replica
          }
          fence_proxy_async_smem();
          named_bar_sync(1, kClipTileUnits);
          if (threadIdx.x == 0) {
            const uint32_t bytes = units * kUnitBytes;
            const size_t li = (t - s0) * E;
            for (int i = 0; i < nstreams; ++i) bulk_s2g(epi.stream(i) + li, slot + (size_t)i * kStreamBytes, bytes);
            bulk_commit();
            if (prev_s >= 0) {
              bulk_wait_read<1>();   // the previous tile's stores have read their slot
              mbar_arrive(&sm->empty[prev_s]);
            }
            prev_s = s;
          }
          if (++s == stages) {
            s = 0;
            phase ^= 1;
          }
        });
    if (threadIdx.x == 0) {
      bulk_wait<0>();
      fence_proxy_async();
    }
  }
  barrier_peers(pv, channel);
}

template <class F>
cudaError_t dispatch_wire(int wire, F&& f) {
  switch (wire) {
    case WIRE_F32: return f(TagF32{});
    case WIRE_BF16: return f(TagBF16{});
    case WIRE_F16: return f(TagF16{});
    default: return cudaErrorInvalidValue;
  }
}

template <class W, class Epi>
cudaError_t launch_update(const PeerView& pv, const ClipDesc* descs, int ndescs, const ClipState* st, int blocks,
                          int stages, int use_nvls, int channel, cudaStream_t stream) {
  const size_t smem = 128 + (size_t)stages * Epi::kStreams * kClipTileUnits * W::kPerVec * 4;
  if (smem > 227 * 1024) return cudaErrorInvalidValue;
  cudaError_t err =
      cudaFuncSetAttribute(clip_update_kernel<W, Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (err != cudaSuccess) return err;
  clip_update_kernel<W, Epi><<<blocks, kClipThreads, smem, stream>>>(pv, descs, ndescs, st, use_nvls, stages, channel);
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_clip_reduce_sumsq(const PeerView& pv, int wire, size_t off, size_t nelem, float scale,
                                     double* slots, const OptHParams* hp, const LaunchCfg& cfg, cudaStream_t stream) {
  if (cfg.blocks < 1 || cfg.blocks > kClipSlotsPerBucket || (off & 15) || (nelem & 7) || (cfg.threads & 31) ||
      cfg.threads < 32 || cfg.threads > 512)
    return cudaErrorInvalidValue;
  return dispatch_wire(wire, [&](auto w) {
    using W = decltype(w);
    clip_reduce_sumsq_kernel<W><<<cfg.blocks, cfg.threads, 0, stream>>>(pv, off, nelem / 8, scale, slots, hp,
                                                                         cfg.use_nvls, cfg.channel);
    return cudaGetLastError();
  });
}

cudaError_t launch_clip_finalize(const PeerView& pv, const double* slots, int nslots, size_t publish_off,
                                 ClipState* state, int channel, cudaStream_t stream) {
  if (nslots < 0 || (publish_off & 15) || pv.world > 256) return cudaErrorInvalidValue;
  clip_finalize_kernel<<<1, 256, 0, stream>>>(pv, slots, nslots, publish_off, state, channel);
  return cudaGetLastError();
}

cudaError_t launch_clip_update(const PeerView& pv, int wire, int opt_kind, const ClipDesc* descs, int ndescs,
                               const ClipState* state, int blocks, int stages, int use_nvls, int channel,
                               cudaStream_t stream) {
  if (blocks < 1 || blocks > kMaxBlocks || ndescs < 1 || stages < 2 || stages > kClipMaxStages ||
      (opt_kind != OPT_SGD && opt_kind != OPT_ADAM))
    return cudaErrorInvalidValue;
  return dispatch_wire(wire, [&](auto w) {
    using W = decltype(w);
    if (opt_kind == OPT_SGD) return launch_update<W, EpiSGD>(pv, descs, ndescs, state, blocks, stages, use_nvls,
                                                             channel, stream);
    return launch_update<W, EpiAdam>(pv, descs, ndescs, state, blocks, stages, use_nvls, channel, stream);
  });
}

}  // namespace bps
