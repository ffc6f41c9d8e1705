// Further kernel families (compression, local optimizers, copies) register
// their bindings from their own translation units.
#pragma once
#include <pybind11/pybind11.h>

void bind_cuda_ext(pybind11::module_& m);
void bind_cuda_ring(pybind11::module_& m);
void bind_cuda_compress(pybind11::module_& m);
void bind_cuda_clip(pybind11::module_& m);
