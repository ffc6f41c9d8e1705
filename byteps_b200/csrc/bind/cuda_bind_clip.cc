// pybind11 surface of the gradient-clipping exchange (kernels/pushpull_clip.cu).
#include <cuda_runtime_api.h>
#include <pybind11/pybind11.h>

#include <stdexcept>
#include <string>

#include "bind/cuda_bind_ext.h"
#include "kernels/pushpull_clip.cuh"

namespace py = pybind11;
using namespace bps;

namespace {
void chk(cudaError_t e, const char* what) {
  if (e != cudaSuccess) throw std::runtime_error(std::string(what) + ": " + cudaGetErrorString(e));
}
}  // namespace

void bind_cuda_clip(py::module_& m) {
  m.attr("CLIP_DESC_BYTES") = (int)sizeof(ClipDesc);
  m.attr("CLIP_STATE_BYTES") = (int)sizeof(ClipState);
  m.attr("CLIP_SLOTS_PER_BUCKET") = kClipSlotsPerBucket;
  m.attr("CLIP_PUBLISH_BYTES") = (int)kClipPublishBytes;

  m.def(
      "clip_reduce_sumsq",
      [](const PeerView& pv, int wire, size_t off, size_t nelem, float scale, uintptr_t slots, uintptr_t hp,
         int blocks, int threads, int channel, bool nvls, uintptr_t stream) {
        LaunchCfg c{blocks, threads, channel, nvls ? 1 : 0, 0, 1};
        chk(launch_clip_reduce_sumsq(pv, wire, off, nelem, scale, (double*)slots, (const OptHParams*)hp, c,
                                     (cudaStream_t)stream),
            "clip_reduce_sumsq");
      },
      py::arg("view"), py::arg("wire"), py::arg("off"), py::arg("nelem"), py::arg("scale"), py::arg("slots"),
      py::arg("hp"), py::arg("blocks"), py::arg("threads") = 512, py::arg("channel") = 0, py::arg("nvls") = false,
      py::arg("stream") = 0,
      "Phase 1: reduce-scatter my shard of the window, scaled, in place; per-CTA sums of squares into slots");

  m.def(
      "clip_finalize",
      [](const PeerView& pv, uintptr_t slots, int nslots, size_t publish_off, uintptr_t state, int channel,
         uintptr_t stream) {
        chk(launch_clip_finalize(pv, (const double*)slots, nslots, publish_off, (ClipState*)state, channel,
                                 (cudaStream_t)stream),
            "clip_finalize");
      },
      py::arg("view"), py::arg("slots"), py::arg("nslots"), py::arg("publish_off"), py::arg("state"),
      py::arg("channel") = 0, py::arg("stream") = 0,
      "Phase 2: global norm and clip coefficient, bit-identical on every rank");

  m.def(
      "clip_update",
      [](const PeerView& pv, int wire, int opt_kind, uintptr_t descs, int ndescs, uintptr_t state, int blocks,
         int stages, bool nvls, int channel, uintptr_t stream) {
        chk(launch_clip_update(pv, wire, opt_kind, (const ClipDesc*)descs, ndescs, (const ClipState*)state, blocks,
                               stages, nvls ? 1 : 0, channel, (cudaStream_t)stream),
            "clip_update");
      },
      py::arg("view"), py::arg("wire"), py::arg("opt_kind"), py::arg("descs"), py::arg("ndescs"), py::arg("state"),
      py::arg("blocks"), py::arg("stages") = 4, py::arg("nvls") = false, py::arg("channel") = 0,
      py::arg("stream") = 0,
      "Phase 3: clipped SGD/Adam update of my shards + parameter all-gather over a table of ClipDesc");
}
