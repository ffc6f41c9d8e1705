// pybind11 surface of the sm_100a extension (module byteps_b200._cuda).
// Tensors cross the boundary as raw device pointers + CUDA stream handles, so
// this module needs no torch headers and rebuilds in seconds.
#include <cuda_runtime_api.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <cstring>
#include <stdexcept>

#include "bind/cuda_bind_ext.h"
#include "comm/symm_mem.h"
#include "kernels/pushpull.cuh"

namespace py = pybind11;
using namespace bps;

namespace {

void check(cudaError_t e, const char* what) {
  if (e != cudaSuccess) throw std::runtime_error(std::string(what) + ": " + cudaGetErrorString(e));
}

LaunchCfg make_cfg(int blocks, int threads, int channel, bool nvls, bool one_shot, bool end_barrier) {
  LaunchCfg c;
  c.blocks = blocks;
  c.threads = threads;
  c.channel = channel;
  c.use_nvls = nvls ? 1 : 0;
  c.one_shot = one_shot ? 1 : 0;
  c.end_barrier = end_barrier ? 1 : 0;
  return c;
}

PeerView make_view(const std::vector<uintptr_t>& data, const std::vector<uintptr_t>& sig, uintptr_t mc,
                   uintptr_t epoch, int rank, int world) {
  if ((int)data.size() != world || (int)sig.size() != world || world < 1 || world > kMaxRanks)
    throw std::runtime_error("PeerView: need `world` data and sig pointers");
  PeerView pv;
  memset(&pv, 0, sizeof(pv));
  for (int r = 0; r < world; ++r) {
    pv.data[r] = (char*)data[r];
    pv.sig[r] = (uint32_t*)sig[r];
  }
  pv.mc_data = (char*)mc;
  pv.epoch = (uint32_t*)epoch;
  pv.rank = rank;
  pv.world = world;
  return pv;
}

}  // namespace

PYBIND11_MODULE(_cuda, m) {
  m.doc() = "byteps_b200 sm_100a kernels + symmetric memory";
  m.attr("MAX_RANKS") = kMaxRanks;
  m.attr("MAX_BLOCKS") = kMaxBlocks;
  m.attr("SIG_BYTES") = kSigBytes;
  m.attr("SIGNAL_PAD_BYTES") = (size_t)kSignalPadBytes;
  m.attr("WIRE_F32") = (int)WIRE_F32;
  m.attr("WIRE_BF16") = (int)WIRE_BF16;
  m.attr("WIRE_F16") = (int)WIRE_F16;
  m.attr("OPT_SGD") = (int)OPT_SGD;
  m.attr("OPT_ADAM") = (int)OPT_ADAM;
  m.attr("SEG_DESC_BYTES") = (int)sizeof(SegDesc);
  m.attr("OPT_HPARAMS_BYTES") = (int)sizeof(OptHParams);

  py::class_<PeerView>(m, "PeerView")
      .def(py::init(&make_view), py::arg("data"), py::arg("sig"), py::arg("mc") = 0, py::arg("epoch") = 0,
           py::arg("rank") = 0, py::arg("world") = 1)
      .def_property_readonly("rank", [](const PeerView& v) { return v.rank; })
      .def_property_readonly("world", [](const PeerView& v) { return v.world; })
      .def_property_readonly("has_mc", [](const PeerView& v) { return v.mc_data != nullptr; })
      .def_property_readonly("epoch_ptr", [](const PeerView& v) { return (uintptr_t)v.epoch; })
      .def_property_readonly("mc_ptr", [](const PeerView& v) { return (uintptr_t)v.mc_data; })
      .def("data_ptr", [](const PeerView& v, int r) { return (uintptr_t)v.data[r]; })
      .def("sig_ptr", [](const PeerView& v, int r) { return (uintptr_t)v.sig[r]; });

  py::class_<SymmMem>(m, "SymmMem")
      .def(py::init<int, int, int, size_t, const std::string&, const std::string&>(), py::arg("rank"),
           py::arg("world"), py::arg("device"), py::arg("data_bytes"), py::arg("mode") = "auto",
           py::arg("token") = "0")
      .def_property_readonly("mode", &SymmMem::mode)
      .def("export_info", [](const SymmMem& s) { return py::bytes(s.export_info()); })
      .def("import_peers",
           [](SymmMem& s, const std::vector<py::bytes>& infos) {
             std::vector<std::string> v;
             for (auto& b : infos) v.push_back(std::string(b));
             py::gil_scoped_release r;
             s.import_peers(v);
           })
      .def("mc_supported", &SymmMem::mc_supported)
      .def("mc_create", [](SymmMem& s) { return py::bytes(s.mc_create()); })
      .def("mc_join",
           [](SymmMem& s, const py::bytes& info) {
             std::string i(info);
             py::gil_scoped_release r;
             s.mc_join(i);
           })
      .def("mc_bind", &SymmMem::mc_bind)
      .def("has_multicast", &SymmMem::has_multicast)
      .def("view", &SymmMem::view)
      .def("local_ptr", [](const SymmMem& s) { return (uintptr_t)s.local_ptr(); })
      .def("peer_ptr", [](const SymmMem& s, int r) { return (uintptr_t)s.peer_ptr(r); })
      .def("mc_ptr", [](const SymmMem& s) { return (uintptr_t)s.mc_ptr(); })
      .def_property_readonly("data_bytes", &SymmMem::data_bytes)
      .def_property_readonly("alloc_bytes", &SymmMem::alloc_bytes)
      .def_property_readonly("rank", &SymmMem::rank)
      .def_property_readonly("world", &SymmMem::world)
      .def("close_server", &SymmMem::close_server);

  m.def(
      "pushpull_inplace",
      [](const PeerView& pv, int wire, size_t off, size_t nelem, float scale, int blocks, int threads, int channel,
         bool nvls, uintptr_t stream) {
        check(launch_pushpull_inplace(pv, wire, off, nelem, scale, make_cfg(blocks, threads, channel, nvls, false, true),
                                      (cudaStream_t)stream),
              "pushpull_inplace");
      },
      py::arg("view"), py::arg("wire"), py::arg("off"), py::arg("nelem"), py::arg("scale"), py::arg("blocks"),
      py::arg("threads") = 512, py::arg("channel") = 0, py::arg("nvls") = false, py::arg("stream") = 0);

  m.def(
      "pushpull_inplace_tma",
      [](const PeerView& pv, int wire, size_t off, size_t nelem, float scale, int blocks, int stages, int channel,
         uintptr_t stream) {
        check(launch_pushpull_inplace_tma(pv, wire, off, nelem, scale, blocks, stages, channel, (cudaStream_t)stream),
              "pushpull_inplace_tma");
      },
      py::arg("view"), py::arg("wire"), py::arg("off"), py::arg("nelem"), py::arg("scale"), py::arg("blocks"),
      py::arg("stages") = 4, py::arg("channel") = 0, py::arg("stream") = 0);

  m.def(
      "reduce_scatter",
      [](const PeerView& pv, int wire, size_t off, size_t nelem, int blocks, int threads, int channel, bool nvls,
         uintptr_t stream) {
        check(launch_reduce_scatter(pv, wire, off, nelem, make_cfg(blocks, threads, channel, nvls, false, true),
                                    (cudaStream_t)stream),
              "reduce_scatter");
      },
      py::arg("view"), py::arg("wire"), py::arg("off"), py::arg("nelem"), py::arg("blocks"), py::arg("threads") = 512,
      py::arg("channel") = 0, py::arg("nvls") = false, py::arg("stream") = 0);

  m.def(
      "all_gather",
      [](const PeerView& pv, int wire, size_t off, size_t nelem, float scale, int blocks, int threads, int channel,
         bool nvls, uintptr_t stream) {
        check(launch_all_gather(pv, wire, off, nelem, scale, make_cfg(blocks, threads, channel, nvls, false, true),
                                (cudaStream_t)stream),
              "all_gather");
      },
      py::arg("view"), py::arg("wire"), py::arg("off"), py::arg("nelem"), py::arg("scale"), py::arg("blocks"),
      py::arg("threads") = 512, py::arg("channel") = 0, py::arg("nvls") = false, py::arg("stream") = 0);

  m.def(
      "pushpull_packed",
      [](const PeerView& pv, int user_dtype, int wire, uintptr_t segs, int nsegs, size_t stage_off, size_t total_elems,
         float scale, int blocks, int threads, int channel, bool nvls, bool one_shot, bool end_barrier,
         uintptr_t stream) {
        check(launch_pushpull_packed(pv, user_dtype, wire, (const SegDesc*)segs, nsegs, stage_off, total_elems, scale,
                                     make_cfg(blocks, threads, channel, nvls, one_shot, end_barrier),
                                     (cudaStream_t)stream),
              "pushpull_packed");
      },
      py::arg("view"), py::arg("user_dtype"), py::arg("wire"), py::arg("segs"), py::arg("nsegs"),
      py::arg("stage_off"), py::arg("total_elems"), py::arg("scale"), py::arg("blocks"), py::arg("threads") = 512,
      py::arg("channel") = 0, py::arg("nvls") = false, py::arg("one_shot") = false, py::arg("end_barrier") = true,
      py::arg("stream") = 0);

  m.def(
      "pushpull_fused_opt",
      [](const PeerView& pv, int grad_dtype, int wire, int param_dtype, int opt_kind, uintptr_t segs, int nsegs,
         size_t stage_off, size_t param_off, size_t total_elems, float scale, uintptr_t master, uintptr_t state0,
         uintptr_t state1, uintptr_t hp, int blocks, int threads, int channel, bool nvls, uintptr_t stream) {
        check(launch_pushpull_fused_opt(pv, grad_dtype, wire, param_dtype, opt_kind, (const SegDesc*)segs, nsegs,
                                        stage_off, param_off, total_elems, scale, (float*)master, (float*)state0,
                                        (float*)state1, (const OptHParams*)hp,
                                        make_cfg(blocks, threads, channel, nvls, false, true), (cudaStream_t)stream),
              "pushpull_fused_opt");
      },
      py::arg("view"), py::arg("grad_dtype"), py::arg("wire"), py::arg("param_dtype"), py::arg("opt_kind"),
      py::arg("segs"), py::arg("nsegs"), py::arg("stage_off"), py::arg("param_off"), py::arg("total_elems"),
      py::arg("scale"), py::arg("master"), py::arg("state0"), py::arg("state1"), py::arg("hp"), py::arg("blocks"),
      py::arg("threads") = 512, py::arg("channel") = 0, py::arg("nvls") = false, py::arg("stream") = 0);

  m.def(
      "pushpull_fused_opt_tma",
      [](const PeerView& pv, int wire, int opt_kind, size_t grad_off, size_t param_off, size_t total_elems,
         float scale, uintptr_t master, uintptr_t state0, uintptr_t state1, uintptr_t hp, int blocks, int stages,
         bool nvls, int channel, uintptr_t stream) {
        check(launch_pushpull_fused_opt_tma(pv, wire, opt_kind, grad_off, param_off, total_elems, scale,
                                            (float*)master, (float*)state0, (float*)state1, (const OptHParams*)hp,
                                            blocks, stages, nvls ? 1 : 0, channel, (cudaStream_t)stream),
              "pushpull_fused_opt_tma");
      },
      py::arg("view"), py::arg("wire"), py::arg("opt_kind"), py::arg("grad_off"), py::arg("param_off"),
      py::arg("total_elems"), py::arg("scale"), py::arg("master"), py::arg("state0"), py::arg("state1"),
      py::arg("hp"), py::arg("blocks"), py::arg("stages") = 4, py::arg("nvls") = false, py::arg("channel") = 0,
      py::arg("stream") = 0,
      "Fused optimizer exchange with TMA-streamed optimizer state (gradients already in the arena)");

  m.def(
      "barrier",
      [](const PeerView& pv, int blocks, int channel, uintptr_t stream) {
        check(launch_barrier(pv, blocks, channel, (cudaStream_t)stream), "barrier");
      },
      py::arg("view"), py::arg("blocks") = 1, py::arg("channel") = 0, py::arg("stream") = 0);

  m.def("shard_units", [](size_t total_units, int world, int rank) {
    size_t b, e;
    shard_units(total_units, world, rank, &b, &e);
    return py::make_tuple(b, e);
  });

  bind_cuda_ext(m);
  bind_cuda_ring(m);
  bind_cuda_compress(m);
  bind_cuda_clip(m);
}
