// shim_module.cc -- python bindings of hoomd_shim (TEST BUILD ONLY).
// HOOMD-blue is not in this image, so the plugin glue under plugin/src is compiled against
// hoomd_shim and exercised through this module: it plays the part of hoomd._hoomd / hoomd.md._md
// (SystemDefinition, ForceCompute, Variant, ParticleGroup, ComputeThermo, Thermostat).  A real
// deployment never builds this file (plugin/CMakeLists.txt).
#include "hoomd/ShimCore.h"
#include "hoomd/md/IntegrationMethodTwoStep.h"
#include "hoomd/md/Thermostat.h"

#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

namespace py = pybind11;
using namespace hoomd;

namespace
    {
template<class T, int W> void fill(const GPUArray<T>& arr, py::array_t<double, py::array::c_style | py::array::forcecast> a, unsigned int N)
    {
    if ((size_t)a.size() != (size_t)N * W)
        throw std::runtime_error("hoomd_shim: array of the wrong size");
    ArrayHandle<T> h(arr, access_location::host, access_mode::overwrite);
    std::memcpy((void*)h.data, a.data(), sizeof(double) * (size_t)N * W);
    }
template<class T, int W> py::array_t<double> fetch(const GPUArray<T>& arr, unsigned int N)
    {
    ArrayHandle<T> h(arr, access_location::host, access_mode::read);
    py::array_t<double> out({(py::ssize_t)N, (py::ssize_t)W});
    std::memcpy(out.mutable_data(), (const void*)h.data, sizeof(double) * (size_t)N * W);
    return out;
    }

struct PublicThermostat : public md::Thermostat
    {
    using md::Thermostat::Thermostat;
    };
    } // namespace

PYBIND11_MODULE(_hoomd_shim, m)
    {
    py::class_<ExecutionConfiguration, std::shared_ptr<ExecutionConfiguration>>(m, "ExecutionConfiguration")
        .def(py::init<bool, int>(), py::arg("gpu") = false, py::arg("gpu_id") = 0)
        .def("isCUDAEnabled", &ExecutionConfiguration::isCUDAEnabled);

    py::class_<ParticleData, std::shared_ptr<ParticleData>>(m, "ParticleData")
        .def(py::init([](unsigned int N, double Lx, double Ly, double Lz, std::vector<std::string> types,
                         std::shared_ptr<ExecutionConfiguration> exec)
                      { return std::make_shared<ParticleData>(N, BoxDim(Lx, Ly, Lz), types, exec); }))
        .def("getN", &ParticleData::getN)
        .def("getTypeByName", &ParticleData::getTypeByName)
        .def("setPositions", [](ParticleData& p, py::array_t<double, py::array::c_style | py::array::forcecast> a)
             { fill<Scalar4, 4>(p.getPositions(), a, p.getN()); })
        .def("setVelocities", [](ParticleData& p, py::array_t<double, py::array::c_style | py::array::forcecast> a)
             { fill<Scalar4, 4>(p.getVelocities(), a, p.getN()); })
        .def("setCharges", [](ParticleData& p, py::array_t<double, py::array::c_style | py::array::forcecast> a)
             { fill<Scalar, 1>(p.getCharges(), a, p.getN()); })
        .def("setImages",
             [](ParticleData& p, py::array_t<int, py::array::c_style | py::array::forcecast> a)
             {
                 if ((size_t)a.size() != (size_t)p.getN() * 3)
                     throw std::runtime_error("hoomd_shim: image array of the wrong size");
                 ArrayHandle<int3> h(p.getImages(), access_location::host, access_mode::overwrite);
                 std::memcpy((void*)h.data, a.data(), sizeof(int) * 3 * (size_t)p.getN());
             })
        .def("setNetForce", [](ParticleData& p, py::array_t<double, py::array::c_style | py::array::forcecast> a)
             { fill<Scalar4, 4>(p.getNetForce(), a, p.getN()); })
        .def("getImages",
             [](ParticleData& p)
             {
                 ArrayHandle<int3> h(p.getImages(), access_location::host, access_mode::read);
                 py::array_t<int> out({(py::ssize_t)p.getN(), (py::ssize_t)3});
                 std::memcpy(out.mutable_data(), (const void*)h.data, sizeof(int) * 3 * (size_t)p.getN());
                 return out;
             })
        .def("getVelocities", [](ParticleData& p) { return fetch<Scalar4, 4>(p.getVelocities(), p.getN()); })
        .def("getPositions", [](ParticleData& p) { return fetch<Scalar4, 4>(p.getPositions(), p.getN()); })
        .def("getTags",
             [](ParticleData& p)
             {
                 ArrayHandle<unsigned int> h(p.getTags(), access_location::host, access_mode::read);
                 return std::vector<unsigned int>(h.data, h.data + p.getN());
             })
        // what HOOMD's particle sorter does (ShimCore.h): the particle now at index j is the one that was at order[j]
        .def("sortParticles", &ParticleData::sortParticles);

    py::class_<SystemDefinition, std::shared_ptr<SystemDefinition>>(m, "SystemDefinition")
        .def(py::init<std::shared_ptr<ParticleData>, uint16_t>(), py::arg("pdata"), py::arg("seed") = 0)
        .def("getParticleData", &SystemDefinition::getParticleData)
        .def("setSeed", &SystemDefinition::setSeed)
        .def("getSeed", &SystemDefinition::getSeed);

    py::class_<ForceCompute, std::shared_ptr<ForceCompute>>(m, "ForceCompute")
        .def("compute", &ForceCompute::compute)
        .def("calcEnergySum", &ForceCompute::calcEnergySum)
        .def("getForces", [](ForceCompute& f)
             { return fetch<Scalar4, 4>(f.getForceArray(), (unsigned int)f.getForceArray().getNumElements()); });

    py::class_<Variant, std::shared_ptr<Variant>>(m, "Variant").def("__call__", &Variant::operator());
    py::class_<VariantConstant, Variant, std::shared_ptr<VariantConstant>>(m, "VariantConstant")
        .def(py::init<Scalar>())
        .def_property("value", &VariantConstant::getValue, &VariantConstant::setValue);

    py::class_<ParticleGroup, std::shared_ptr<ParticleGroup>>(m, "ParticleGroup")
        .def(py::init<std::shared_ptr<SystemDefinition>, const std::vector<unsigned int>&>())
        .def("getNumMembers", &ParticleGroup::getNumMembers)
        .def("setTranslationalDOF", &ParticleGroup::setTranslationalDOF)
        .def("setRotationalDOF", &ParticleGroup::setRotationalDOF)
        .def("getTranslationalDOF", &ParticleGroup::getTranslationalDOF);

    py::class_<md::ComputeThermo, std::shared_ptr<md::ComputeThermo>>(m, "ComputeThermo")
        .def(py::init<std::shared_ptr<SystemDefinition>, std::shared_ptr<ParticleGroup>>())
        .def("compute", &md::ComputeThermo::compute)
        .def("getTranslationalKineticEnergy", &md::ComputeThermo::getTranslationalKineticEnergy)
        .def("setRotationalKineticEnergy", &md::ComputeThermo::setRotationalKineticEnergy);

    py::class_<md::IntegrationMethodTwoStep, std::shared_ptr<md::IntegrationMethodTwoStep>>(m, "IntegrationMethodTwoStep")
        .def("integrateStepOne", &md::IntegrationMethodTwoStep::integrateStepOne)
        .def("integrateStepTwo", &md::IntegrationMethodTwoStep::integrateStepTwo)
        .def("setDeltaT", &md::IntegrationMethodTwoStep::setDeltaT);

    py::class_<md::Thermostat, std::shared_ptr<md::Thermostat>>(m, "Thermostat")
        .def("getRescalingFactorsOne", &md::Thermostat::getRescalingFactorsOne)
        .def("getRescalingFactorsTwo", &md::Thermostat::getRescalingFactorsTwo);

    // the draws the next RandomGenerator will hand out (HOOMD's RNG is upstream code, see ShimCore.h)
    m.def("inject_draws",
          [](std::vector<double> v)
          {
              auto& q = RandomGenerator::injected();
              q.clear();
              for (double x : v)
                  q.push_back(x);
          });
    }
