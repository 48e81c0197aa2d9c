// CavityForceComputeGPU.cc -- see the header.  No CPU fallback: a failure of the CUDA path throws.
#include "CavityForceComputeGPU.h"

#include <cuda_runtime.h>
#include <pybind11/numpy.h>

#include <algorithm>
#include <stdexcept>
#include <string>
#include <vector>

namespace hoomd
    {
namespace cavitymd
    {
namespace
    {
void check(int err, const char* what)
    {
    if (err == 702) // cudaErrorLaunchTimeout: see include/cavb200.h, conventions
        throw std::runtime_error(std::string("CavityForceComputeGPU: ") + what
                                 + ": an earlier cavity-force kernel could not run with its whole grid resident (the GPU is "
                                   "shared with another stream or process), so that step's forces were not written; the force "
                                   "now uses cooperative launches");
    if (err != 0)
        throw std::runtime_error(std::string("CavityForceComputeGPU: ") + what + ": " + cavb200_error_string(err));
    }
    } // namespace

CavityForceComputeGPU::CavityForceComputeGPU(std::shared_ptr<SystemDefinition> sysdef, Scalar omegac, Scalar couplstr,
                                             Scalar phmass)
    : ForceCompute(sysdef), m_handle(nullptr), m_fresh(true)
    {
    m_exec_conf->msg->notice(5) << "Constructing CavityForceComputeGPU (cavb200)" << std::endl;
    if (!m_exec_conf->isCUDAEnabled())
        throw std::runtime_error("CavityForceComputeGPU requires a GPU execution configuration (no CPU fallback)");
#ifdef ENABLE_MPI
    // the dipole is summed over THIS rank's particles only (like the reference, SURVEY.md Appendix C #12): refuse
    // rather than compute a wrong force under domain decomposition
    if (m_sysdef->isDomainDecomposed())
        throw std::runtime_error("CavityForceComputeGPU (cavb200): domain-decomposed (multi-rank) runs are not supported");
#endif
    setParams(omegac, couplstr, phmass);
    for (int k = 0; k < 3; k++)
        m_energies[k] = m_dipole[k] = 0.0;
    int device = 0;
#ifdef ENABLE_HIP
    cudaGetDevice(&device);
#endif
    check(cavb200_create(&m_handle, device), "cavb200_create");
    }

CavityForceComputeGPU::~CavityForceComputeGPU()
    {
    m_exec_conf->msg->notice(5) << "Destroying CavityForceComputeGPU" << std::endl;
    cavb200_destroy(m_handle);
    }

void CavityForceComputeGPU::setParams(Scalar omegac, Scalar couplstr, Scalar phmass)
    {
    m_params.omegac = omegac;
    m_params.couplstr = couplstr;
    m_params.phmass = phmass;
    m_params.K = phmass * omegac * omegac; // reference src/CavityForceCompute.h:38-42
    }

pybind11::dict CavityForceComputeGPU::getParams()
    {
    pybind11::dict v;
    v["omegac"] = m_params.omegac;
    v["couplstr"] = m_params.couplstr;
    v["K"] = m_params.K;
    v["phmass"] = m_params.phmass;
    return v;
    }

void CavityForceComputeGPU::useHandle(cavb200_handle* h, int mode)
    {
    if (mode != 0 && !h)
        throw std::runtime_error("CavityForceComputeGPU::useHandle: rank-1 modes need the integration method's handle");
    m_ext_handle = mode ? h : nullptr;
    m_mode = mode;
    m_integrator_reduced = false;
    m_zeroed = false;
    m_fresh = false;
    }

void CavityForceComputeGPU::computeForces(uint64_t timestep)
    {
    (void)timestep;
    const unsigned int N = m_pdata->getN();
    if (m_mode == 2 && m_integrator_reduced)
        return; // the integration method's step one has already reduced the dipole of these positions
    // 'L' missing from the type list: the reference GPU class reports zero energies and leaves the
    // forces zero (src/CavityForceComputeGPU.cc:114-123); UINT32_MAX asks the library for exactly that
    uint32_t L_typeid = 0xFFFFFFFFu;
    try
        {
        L_typeid = m_pdata->getTypeByName("L");
        }
    catch (...)
        {
        }
    const BoxDim box = m_pdata->getGlobalBox();
    const Scalar3 L = box.getL();

    ArrayHandle<Scalar4> d_pos(m_pdata->getPositions(), access_location::device, access_mode::read);
    ArrayHandle<Scalar> d_charge(m_pdata->getCharges(), access_location::device, access_mode::read);
    ArrayHandle<int3> d_image(m_pdata->getImages(), access_location::device, access_mode::read);
    if (m_mode != 0)
        {
        // rank-1: the contribution to HOOMD's net force is zero (m_force was zero-initialised by ForceCompute and is
        // zeroed once here in case the object ran in stored mode before); Dq / F_L stay on the method's handle
        if (!m_zeroed)
            {
            ArrayHandle<Scalar4> d_f(m_force, access_location::device, access_mode::overwrite);
            cudaMemsetAsync(d_f.data, 0, sizeof(Scalar4) * (size_t)N, (cudaStream_t)m_stream);
            m_zeroed = true;
            }
        check(cavb200_force_rank1(m_ext_handle, reinterpret_cast<const double*>(d_pos.data), d_charge.data,
                                  reinterpret_cast<const int32_t*>(d_image.data), N, L.x, L.y, L.z, L_typeid, &m_params,
                                  m_stream),
              "cavb200_force_rank1");
        m_fresh = false;
        return;
        }
    ArrayHandle<Scalar4> d_force(m_force, access_location::device, access_mode::overwrite);

    // HOOMD runs its kernels on the legacy default stream: stream 0 ordering is the contract
    check(cavb200_force(m_handle, reinterpret_cast<const double*>(d_pos.data), d_charge.data,
                        reinterpret_cast<const int32_t*>(d_image.data), reinterpret_cast<double*>(d_force.data), N, L.x,
                        L.y, L.z, L_typeid, &m_params, m_stream),
          "cavb200_force");
    m_fresh = false; // no synchronisation here: energies are fetched when somebody asks
    }

void CavityForceComputeGPU::readBack()
    {
    if (m_fresh)
        return;
    int32_t photon = -1;
    check(cavb200_force_read(m_ext_handle ? m_ext_handle : m_handle, m_energies, m_dipole, &photon, m_stream),
          "cavb200_force_read");
    m_fresh = true;
    }

Scalar CavityForceComputeGPU::getHarmonicEnergy()
    {
    readBack();
    return m_energies[0];
    }
Scalar CavityForceComputeGPU::getCouplingEnergy()
    {
    readBack();
    return m_energies[1];
    }
Scalar CavityForceComputeGPU::getDipoleSelfEnergy()
    {
    readBack();
    return m_energies[2];
    }
bool CavityForceComputeGPU::getCooperativeLaunch() const
    {
    int pdl = 1;
    cavb200_get_tuning(m_handle, "pdl", &pdl);
    return pdl == 0;
    }
void CavityForceComputeGPU::setCooperativeLaunch(bool c) { cavb200_set_tuning(m_handle, "pdl", c ? 0 : 1); }
unsigned long long CavityForceComputeGPU::getFaultCount() const { return cavb200_fault_count(m_handle); }

pybind11::tuple CavityForceComputeGPU::getDipole()
    {
    readBack();
    return pybind11::make_tuple(m_dipole[0], m_dipole[1], m_dipole[2]);
    }

void CavityForceComputeGPU::trackOpen(unsigned int capacity)
    {
    check(cavb200_track_open(m_handle, capacity), "cavb200_track_open");
    }

void CavityForceComputeGPU::trackSetReference()
    {
    check(cavb200_track_set_reference_from(m_handle, m_ext_handle ? m_ext_handle : m_handle, m_stream),
          "cavb200_track_set_reference_from");
    }

void CavityForceComputeGPU::trackRecord(uint64_t timestep)
    {
    // asynchronous, ordered after this step's kernels on HOOMD's stream; the photon's kinetic energy needs the
    // velocities, everything else is already on the device: the force result on the handle that computed it, KE / alpha
    // on the handle the thermostat ran on
    ArrayHandle<Scalar4> d_vel(m_pdata->getVelocities(), access_location::device, access_mode::read);
    check(cavb200_track_record_from(m_handle, m_ext_handle ? m_ext_handle : m_handle, m_bussi_handle, timestep,
                                    reinterpret_cast<const double*>(d_vel.data), m_pdata->getN(),
                                    m_vel_pending ? CAVB200_TRACK_VELOCITIES_PENDING : 0u, m_stream),
          "cavb200_track_record_from");
    }

pybind11::list CavityForceComputeGPU::trackRead(unsigned int max_records)
    {
    std::vector<double> buf((size_t)max_records * CAVB200_TRACK_WORDS + 1);
    uint32_t n = 0;
    uint64_t total = 0;
    check(cavb200_track_read(m_handle, buf.data(), max_records, &n, &total, m_stream), "cavb200_track_read");
    pybind11::list out;
    for (uint32_t r = 0; r < n; r++)
        {
        pybind11::tuple row(CAVB200_TRACK_WORDS);
        for (int k = 0; k < CAVB200_TRACK_WORDS; k++)
            row[k] = buf[(size_t)r * CAVB200_TRACK_WORDS + k];
        out.append(row);
        }
    return out;
    }

void CavityForceComputeGPU::fktOpen(pybind11::object kvectors, unsigned int max_references, unsigned int capacity)
    {
    std::vector<double> k;
    for (auto row : kvectors)
        {
        size_t c = 0;
        for (auto v : row)
            {
            k.push_back(v.cast<double>());
            c++;
            }
        if (c != 3)
            throw std::invalid_argument("CavityForceComputeGPU::fktOpen: every wave vector needs 3 components");
        }
    check(cavb200_fkt_track_open(m_handle, k.data(), (uint32_t)(k.size() / 3), max_references, capacity, m_pdata->getN()),
          "cavb200_fkt_track_open");
    m_fkt_words = 2 + max_references + (unsigned int)(k.size() / 3) * 2;
    }

void CavityForceComputeGPU::fktStep(uint64_t timestep, bool record, bool add_reference)
    {
    // asynchronous on this object's stream, after whatever wrote the positions; the wrapped positions of every particle,
    // photon included, as the reference's compute_density_field takes them
    ArrayHandle<Scalar4> d_pos(m_pdata->getPositions(), access_location::device, access_mode::read);
    const uint32_t flags = (record ? CAVB200_FKT_RECORD : 0u) | (add_reference ? CAVB200_FKT_ADD_REFERENCE : 0u);
    check(cavb200_fkt_track_step(m_handle, reinterpret_cast<const double*>(d_pos.data), m_pdata->getN(), timestep, flags,
                                 m_stream),
          "cavb200_fkt_track_step");
    }

pybind11::tuple CavityForceComputeGPU::fktRead(unsigned int max_records)
    {
    const size_t words = m_fkt_words ? m_fkt_words : 1;
    std::vector<double> buf((size_t)max_records * words + 1);
    uint32_t n = 0;
    uint64_t total = 0;
    check(cavb200_fkt_track_read(m_handle, buf.data(), max_records, &n, &total, m_stream), "cavb200_fkt_track_read");
    pybind11::array_t<double> out({(size_t)n, words});
    std::copy(buf.begin(), buf.begin() + (size_t)n * words, out.mutable_data());
    return pybind11::make_tuple(out, total);
    }

namespace detail
    {
void export_CavityForceComputeGPU(pybind11::module& m)
    {
    // same python-visible name, constructor and methods as the reference export
    // (src/CavityForceComputeGPU.cc:257-265 + the base-class methods of src/CavityForceCompute.cc:212-224)
    pybind11::class_<CavityForceComputeGPU, ForceCompute, std::shared_ptr<CavityForceComputeGPU>>(m, "CavityForceComputeGPU")
        .def(pybind11::init<std::shared_ptr<SystemDefinition>, Scalar, Scalar, Scalar>(), pybind11::arg("sysdef"),
             pybind11::arg("omegac"), pybind11::arg("couplstr"), pybind11::arg("phmass") = 1.0)
        .def("setParams", &CavityForceComputeGPU::setParams, pybind11::arg("omegac"), pybind11::arg("couplstr"),
             pybind11::arg("phmass") = 1.0)
        .def("getParams", &CavityForceComputeGPU::getParams)
        .def("getHarmonicEnergy", &CavityForceComputeGPU::getHarmonicEnergy)
        .def("getCouplingEnergy", &CavityForceComputeGPU::getCouplingEnergy)
        .def("getDipoleSelfEnergy", &CavityForceComputeGPU::getDipoleSelfEnergy)
        .def("getDipole", &CavityForceComputeGPU::getDipole)
        .def_property("cooperative_launch", &CavityForceComputeGPU::getCooperativeLaunch,
                      &CavityForceComputeGPU::setCooperativeLaunch)
        .def("getFaultCount", &CavityForceComputeGPU::getFaultCount)
        .def_property("stream", &CavityForceComputeGPU::getStream, &CavityForceComputeGPU::setStream)
        .def("trackOpen", &CavityForceComputeGPU::trackOpen, pybind11::arg("capacity"))
        .def("trackSetReference", &CavityForceComputeGPU::trackSetReference)
        .def("trackRecord", &CavityForceComputeGPU::trackRecord, pybind11::arg("timestep"))
        .def("trackRead", &CavityForceComputeGPU::trackRead, pybind11::arg("max_records"))
        .def("fktOpen", &CavityForceComputeGPU::fktOpen, pybind11::arg("kvectors"), pybind11::arg("max_references"),
             pybind11::arg("capacity"))
        .def("fktStep", &CavityForceComputeGPU::fktStep, pybind11::arg("timestep"), pybind11::arg("record"),
             pybind11::arg("add_reference"))
        .def("fktRead", &CavityForceComputeGPU::fktRead, pybind11::arg("max_records"));
    }
    } // namespace detail
    } // namespace cavitymd
    } // namespace hoomd
