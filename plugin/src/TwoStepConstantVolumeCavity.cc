// TwoStepConstantVolumeCavity.cc -- see the header.  No CPU fallback: a failure of the CUDA path throws.
#include "TwoStepConstantVolumeCavity.h"

#include <cuda_runtime.h>
#include <stdexcept>

namespace hoomd::md
    {
TwoStepConstantVolumeCavity::TwoStepConstantVolumeCavity(std::shared_ptr<SystemDefinition> sysdef,
                                                         std::shared_ptr<ParticleGroup> group,
                                                         std::shared_ptr<Thermostat> thermostat,
                                                         std::shared_ptr<cavitymd::CavityForceComputeGPU> cavity,
                                                         const std::string& mode)
    : IntegrationMethodTwoStep(sysdef, group), m_thermostat(thermostat), m_source(nullptr), m_cavity(cavity),
      m_handle(nullptr), m_started(false), m_pending(false), m_index_list(false), m_group_stale(true), m_use_mask(false),
      m_first(0), m_group_n(0), m_group_N(0), m_photon_stale(false)
    {
    if (!m_exec_conf->isCUDAEnabled())
        throw std::runtime_error("TwoStepConstantVolumeCavity requires a GPU execution configuration (no CPU fallback)");
    if (mode == "stored")
        m_mode = STORED;
    else if (mode == "rank1")
        m_mode = RANK1;
    else if (mode == "one_launch")
        m_mode = ONE_LAUNCH;
    else
        throw std::invalid_argument("TwoStepConstantVolumeCavity: mode must be 'stored', 'rank1' or 'one_launch'");
    if (m_mode != STORED && !m_cavity)
        throw std::invalid_argument("TwoStepConstantVolumeCavity: the rank-1 modes need the CavityForceComputeGPU object");
#ifdef ENABLE_MPI
    if (m_sysdef->isDomainDecomposed())
        throw std::runtime_error("TwoStepConstantVolumeCavity (cavb200): domain-decomposed (multi-rank) runs are not supported");
#endif
    if (m_thermostat)
        {
        m_source = dynamic_cast<CavbBussiSource*>(m_thermostat.get());
        if (!m_source)
            throw std::invalid_argument("TwoStepConstantVolumeCavity: the thermostat must be a BussiReservoirThermostat (or None)");
        }
    int device = 0;
    cudaGetDevice(&device);
    check(cavb200_create(&m_handle, device), "cavb200_create");
    if (m_source)
        m_source->adoptHandle(m_handle);
    if (m_cavity && m_mode != STORED)
        m_cavity->useHandle(m_handle, m_mode == RANK1 ? 1 : 2);
    m_pdata->getParticleSortSignal().connect<TwoStepConstantVolumeCavity, &TwoStepConstantVolumeCavity::slotParticleSort>(this);
    }

TwoStepConstantVolumeCavity::~TwoStepConstantVolumeCavity()
    {
    m_pdata->getParticleSortSignal().disconnect<TwoStepConstantVolumeCavity, &TwoStepConstantVolumeCavity::slotParticleSort>(
        this);
    if (m_source)
        m_source->adoptHandle(nullptr);
    if (m_cavity && m_mode != STORED)
        m_cavity->useHandle(nullptr, 0);
    cavb200_destroy(m_handle);
    }

std::string TwoStepConstantVolumeCavity::getMode() const
    {
    return m_mode == STORED ? "stored" : (m_mode == RANK1 ? "rank1" : "one_launch");
    }

void TwoStepConstantVolumeCavity::check(int err, const char* what) const
    {
    if (err == 702) // cudaErrorLaunchTimeout: include/cavb200.h, conventions
        throw std::runtime_error(std::string("TwoStepConstantVolumeCavity: ") + what
                                 + ": an earlier step's persistent kernel could not run with its whole grid resident (the "
                                   "GPU is shared with another stream or process); that step was not integrated");
    if (err)
        throw std::runtime_error(std::string("TwoStepConstantVolumeCavity: ") + what + ": " + cavb200_error_string(err));
    }

void TwoStepConstantVolumeCavity::window(unsigned int& first, unsigned int& n)
    {
    // the fused kernels thermostat a window of the index space; HOOMD hands out an index list
    n = m_group->getNumMembers();
    first = 0;
    if (n == 0)
        return;
    ArrayHandle<unsigned int> h_idx(m_group->getIndexArray(), access_location::host, access_mode::read);
    first = h_idx.data[0];
    if (h_idx.data[n - 1] != first + (n - 1))
        throw std::runtime_error("TwoStepConstantVolumeCavity: the thermostatted group must be a contiguous index range");
    // (first / last / count identify a range when the list is ascending and free of duplicates, which ParticleGroup's
    // index list is [HOOMD-upstream]; checked in full on the first step)
    if (!m_started)
        for (unsigned int j = 0; j < n; j++)
            if (h_idx.data[j] != first + j)
                throw std::runtime_error("TwoStepConstantVolumeCavity: the thermostatted group must be a contiguous index range");
    }

void TwoStepConstantVolumeCavity::setIndexListGroup(bool on)
    {
    m_index_list = on;
    m_group_stale = true;
    }

void TwoStepConstantVolumeCavity::slotParticleSort()
    {
    m_group_stale = true;
    m_photon_stale = true;
    }

uint32_t TwoStepConstantVolumeCavity::photonTypeId() const
    {
    try
        {
        return m_pdata->getTypeByName("L");
        }
    catch (...)
        {
        return 0xFFFFFFFFu;
        }
    }

void TwoStepConstantVolumeCavity::group(unsigned int& first, unsigned int& n)
    {
    if (!m_index_list)
        {
        window(first, n);
        return;
        }
    n = m_group->getNumMembers();
    const unsigned int N = m_pdata->getN();
    if (m_group_stale || n != m_group_n || N != m_group_N)
        {
        bool contiguous = true;
            {
            ArrayHandle<unsigned int> h_idx(m_group->getIndexArray(), access_location::host, access_mode::read);
            m_first = n ? h_idx.data[0] : 0;
            for (unsigned int j = 0; j < n && contiguous; j++)
                contiguous = h_idx.data[j] == m_first + j;
            }
        m_use_mask = !contiguous;
        if (m_use_mask)
            {
            ArrayHandle<unsigned int> d_idx(m_group->getIndexArray(), access_location::device, access_mode::read);
            check(cavb200_group_set(m_handle, d_idx.data, n, N, nullptr), "cavb200_group_set");
            }
        m_group_n = n;
        m_group_N = N;
        m_group_stale = false;
        }
    first = m_use_mask ? CAVB200_GROUP_MASK : m_first;
    }

void TwoStepConstantVolumeCavity::reindexPhoton(uint32_t L_typeid)
    {
    // the rank-1 kicks give F_L to the particle at the photon index of the last result, which a sort has moved
    if (!m_photon_stale || m_mode == STORED)
        return;
    ArrayHandle<Scalar4> d_pos(m_pdata->getPositions(), access_location::device, access_mode::read);
    check(cavb200_rank1_reindex(m_handle, reinterpret_cast<const double*>(d_pos.data), m_pdata->getN(), L_typeid, nullptr),
          "cavb200_rank1_reindex (the rank-1 modes follow a particle sort with one particle of type 'L' only)");
    m_photon_stale = false;
    }

void TwoStepConstantVolumeCavity::integrateStepOne(uint64_t timestep)
    {
    const unsigned int N = m_pdata->getN();
    if (N == 0)
        return;
    unsigned int first = 0, n = 0;
    group(first, n);
    const uint32_t L_typeid = photonTypeId();
    reindexPhoton(L_typeid);
    const Scalar3 L = m_pdata->getGlobalBox().getL();
    cavb200_bussi_args args = {};
    const cavb200_bussi_args* bussi = nullptr;
    if (m_source && m_deltaT != 0.0)
        {
        args = m_source->drawBussiArgs(timestep, m_deltaT);
        bussi = &args;
        }
    ArrayHandle<Scalar4> d_pos(m_pdata->getPositions(), access_location::device, access_mode::readwrite);
    ArrayHandle<Scalar4> d_vel(m_pdata->getVelocities(), access_location::device, access_mode::readwrite);
    ArrayHandle<int3> d_image(m_pdata->getImages(), access_location::device, access_mode::readwrite);
    ArrayHandle<Scalar4> d_net(m_pdata->getNetForce(), access_location::device, access_mode::read);
    ArrayHandle<Scalar> d_charge(m_pdata->getCharges(), access_location::device, access_mode::read);
    double* pos = reinterpret_cast<double*>(d_pos.data);
    double* vel = reinterpret_cast<double*>(d_vel.data);
    int32_t* image = reinterpret_cast<int32_t*>(d_image.data);
    const double* net = reinterpret_cast<const double*>(d_net.data);

    if (!m_started)
        {
        // the first alpha needs KE(v(t0)): one reduce pass, once (afterwards step two leaves the next KE on the device)
        if (first == CAVB200_GROUP_MASK)
            {
            ArrayHandle<unsigned int> d_idx(m_group->getIndexArray(), access_location::device, access_mode::read);
            check(cavb200_bussi_ke(m_handle, vel, d_idx.data, 0, n, nullptr), "cavb200_bussi_ke");
            }
        else
            check(cavb200_bussi_ke(m_handle, vel, nullptr, first, n, nullptr), "cavb200_bussi_ke");
        m_started = true;
        }
    switch (m_mode)
        {
    case STORED:
        check(cavb200_nvt_step_one_wrap(m_handle, pos, vel, net, image, N, m_deltaT, L.x, L.y, L.z, first, n, bussi, nullptr),
              "cavb200_nvt_step_one_wrap");
        break;
    case RANK1:
        check(cavb200_nvt_step_one_rank1_wrap(m_handle, pos, vel, net, d_charge.data, image, N, m_deltaT, L.x, L.y, L.z,
                                              L_typeid, m_cavity->params().couplstr, first, n, bussi, nullptr),
              "cavb200_nvt_step_one_rank1_wrap");
        break;
    case ONE_LAUNCH:
        if (m_pending)
            check(cavb200_md_step_fused_wrap(m_handle, pos, vel, net, d_charge.data, image, N, m_deltaT, L.x, L.y, L.z,
                                             L_typeid, &m_cavity->params(), first, n, bussi, nullptr),
                  "cavb200_md_step_fused_wrap");
        else
            check(cavb200_md_step_one_wrap(m_handle, pos, vel, net, d_charge.data, image, N, m_deltaT, L.x, L.y, L.z, L_typeid,
                                           &m_cavity->params(), first, n, bussi, nullptr),
                  "cavb200_md_step_one_wrap");
        m_pending = false;
        m_cavity->integratorHasReduced(); // the dipole of the new positions is on the device: compute() has nothing to do
        break;
        }
    }

void TwoStepConstantVolumeCavity::integrateStepTwo(uint64_t timestep)
    {
    (void)timestep;
    const unsigned int N = m_pdata->getN();
    if (N == 0)
        return;
    if (m_mode == ONE_LAUNCH)
        {
        m_pending = true; // rides on the next step one (or flush())
        return;
        }
    unsigned int first = 0, n = 0;
    group(first, n);
    const uint32_t L_typeid = photonTypeId();
    reindexPhoton(L_typeid);
    ArrayHandle<Scalar4> d_vel(m_pdata->getVelocities(), access_location::device, access_mode::readwrite);
    ArrayHandle<Scalar4> d_net(m_pdata->getNetForce(), access_location::device, access_mode::read);
    double* vel = reinterpret_cast<double*>(d_vel.data);
    const double* net = reinterpret_cast<const double*>(d_net.data);
    if (m_mode == STORED)
        {
        check(cavb200_nvt_step_two(m_handle, vel, net, N, m_deltaT, first, n, nullptr), "cavb200_nvt_step_two");
        return;
        }
    ArrayHandle<Scalar4> d_pos(m_pdata->getPositions(), access_location::device, access_mode::read);
    ArrayHandle<Scalar> d_charge(m_pdata->getCharges(), access_location::device, access_mode::read);
    check(cavb200_nvt_step_two_rank1(m_handle, vel, net, d_charge.data, reinterpret_cast<const double*>(d_pos.data), N,
                                     m_deltaT, L_typeid, m_cavity->params().couplstr, first, n, nullptr),
          "cavb200_nvt_step_two_rank1");
    }

void TwoStepConstantVolumeCavity::flush()
    {
    if (m_mode != ONE_LAUNCH || !m_pending)
        return;
    const unsigned int N = m_pdata->getN();
    unsigned int first = 0, n = 0;
    group(first, n);
    const uint32_t L_typeid = photonTypeId();
    reindexPhoton(L_typeid); // the deferred kick forms the rank-1 force from the last result
    ArrayHandle<Scalar4> d_vel(m_pdata->getVelocities(), access_location::device, access_mode::readwrite);
    ArrayHandle<Scalar4> d_net(m_pdata->getNetForce(), access_location::device, access_mode::read);
    ArrayHandle<Scalar4> d_pos(m_pdata->getPositions(), access_location::device, access_mode::read);
    ArrayHandle<Scalar> d_charge(m_pdata->getCharges(), access_location::device, access_mode::read);
    check(cavb200_nvt_step_two_rank1(m_handle, reinterpret_cast<double*>(d_vel.data), reinterpret_cast<const double*>(d_net.data),
                                     d_charge.data, reinterpret_cast<const double*>(d_pos.data), N, m_deltaT, L_typeid,
                                     m_cavity->params().couplstr, first, n, nullptr),
          "cavb200_nvt_step_two_rank1");
    m_pending = false;
    // the velocities are now complete, but the next step one must not redo this half kick: restart from md_step_one
    }

namespace detail
    {
void export_TwoStepConstantVolumeCavity(pybind11::module& m)
    {
    namespace py = pybind11;
    py::class_<TwoStepConstantVolumeCavity, IntegrationMethodTwoStep, std::shared_ptr<TwoStepConstantVolumeCavity>>(
        m, "TwoStepConstantVolumeCavity")
        .def(py::init<std::shared_ptr<SystemDefinition>, std::shared_ptr<ParticleGroup>, std::shared_ptr<Thermostat>,
                      std::shared_ptr<cavitymd::CavityForceComputeGPU>, const std::string&>(),
             py::arg("sysdef"), py::arg("group"), py::arg("thermostat"), py::arg("cavity_force"), py::arg("mode") = "rank1")
        .def("flush", &TwoStepConstantVolumeCavity::flush)
        .def_property_readonly("mode", &TwoStepConstantVolumeCavity::getMode)
        .def_property("index_list_group", &TwoStepConstantVolumeCavity::getIndexListGroup,
                      &TwoStepConstantVolumeCavity::setIndexListGroup)
        .def("getLaunchCount", &TwoStepConstantVolumeCavity::getLaunchCount);
    }
    } // namespace detail
    } // namespace hoomd::md
