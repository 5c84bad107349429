// tests/pyrichdem_module.cpp -- the reference's OWN pybind11 module (`_richdem`), built with the B200 drop-in layer.
//
// This translation unit is the whole "patch" a pyrichdem maintainer needs (INTEGRATION.md section 3a): the explicit
// specialisations of include/richdem_b200.hpp must be visible before the binding code names the templates, so the
// header is included first and the unmodified reference binding source (wrappers/pyrichdem/src/pywrapper.cpp, found
// through -I<reference>/wrappers/pyrichdem/src at compile time; nothing of it is copied into this repository) follows.
// The resulting module serves richdem/__init__.py unchanged: FillDepressions, ResolveFlats, FlowAccumulation and
// FlowProportions on float32 rasters run on the GPU, every other dtype / method keeps the reference's CPU templates.
// Built by oracle/Makefile (`bindings`) into build/reference_bindings/pyrichdem/ (git-ignored).
#include <richdem_b200.hpp>

#include <pywrapper.cpp>
