// _cavitymd: same module name and class name as the reference (reference src/cavitymd/module.cc:27-34).
// This build exports the GPU class only; the CPU class CavityForceCompute stays the reference's own
// file when a CPU device is wanted (plugin/CMakeLists.txt option CAVB200_WITH_REFERENCE_CPU).
#include "CavityForceComputeGPU.h"
#include "TwoStepConstantVolumeCavity.h"
#ifdef HOOMD_SHIM_CORE_H
#include <pybind11/stl.h>
#endif

PYBIND11_MODULE(_cavitymd, m)
    {
    hoomd::cavitymd::detail::export_CavityForceComputeGPU(m);
    // the fused integration method (SURVEY.md 8f.1/8f.2): new functionality, not in the reference's module
    hoomd::md::detail::export_TwoStepConstantVolumeCavity(m);
#ifdef HOOMD_SHIM_CORE_H
    // shim test build only: the photon bath's uniform draws are injected, into this module's own copy of the queue (as
    // _bussi_reservoir._inject_draws does for the thermostat's)
    m.def("_inject_draws",
          [](std::vector<double> v)
          {
              auto& q = hoomd::RandomGenerator::injected();
              q.clear();
              for (double x : v)
                  q.push_back(x);
          });
#endif
    }
