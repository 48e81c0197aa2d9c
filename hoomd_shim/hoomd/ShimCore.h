// hoomd_shim -- a MINIMAL stand-in for the HOOMD-blue headers the cav-hoomd plugin sources use.
//
// HOOMD-blue is not installed in this image (SURVEY.md section 8c), so nothing that includes
// <hoomd/...> can be compiled against the real thing here.  This shim declares exactly the
// symbols that
//   * the reference translation units src/CavityForceCompute.cc and
//     src/BussiReservoirThermostat.h (+ the vendored src/Thermostat.h) use, so that they compile
//     VERBATIM BY PATH into oracle/_ref/ (the parity oracle), and
//   * this repo's plugin glue under plugin/ uses, so that it can be built and exercised on a GPU
//     box without HOOMD.
// It is written from the call sites in those files (SURVEY.md Appendix B lists the assumed
// upstream contracts); it is not derived from HOOMD's sources.  A real deployment compiles
// plugin/ against an installed HOOMD instead (plugin/CMakeLists.txt) and never sees this
// directory.
#ifndef HOOMD_SHIM_CORE_H
#define HOOMD_SHIM_CORE_H

#include <algorithm>
#include <array>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <deque>
#include <iostream>
#include <map>
#include <memory>
#include <sstream>
#include <stdexcept>
#include <string>
#include <vector>

#ifdef ENABLE_HIP
#include <cuda_runtime.h>
#else
struct double2 { double x, y; };
struct double3 { double x, y, z; };
struct alignas(16) double4 { double x, y, z, w; };
struct int3 { int x, y, z; };
struct uint3 { unsigned int x, y, z; };
#endif

#ifndef PYBIND11_EXPORT
#define PYBIND11_EXPORT __attribute__((visibility("default")))
#endif

namespace hoomd
    {
typedef double Scalar;
typedef double LongReal;
typedef double2 Scalar2;
typedef double3 Scalar3;
typedef double4 Scalar4;

inline Scalar3 make_scalar3(Scalar x, Scalar y, Scalar z)
    {
    Scalar3 r;
    r.x = x; r.y = y; r.z = z;
    return r;
    }
inline Scalar4 make_scalar4(Scalar x, Scalar y, Scalar z, Scalar w)
    {
    Scalar4 r;
    r.x = x; r.y = y; r.z = z; r.w = w;
    return r;
    }

// type ids live in the low 32 bits of pos.w (union overlay, SURVEY.md Appendix B)
inline int __scalar_as_int(Scalar s)
    {
    int i;
    std::memcpy(&i, &s, sizeof(int));
    return i;
    }
inline Scalar __int_as_scalar(int i)
    {
    Scalar s = 0.0;
    std::memcpy(&s, &i, sizeof(int));
    return s;
    }

struct access_location { enum Enum { host, device }; };
struct access_mode { enum Enum { read, readwrite, overwrite }; };

//! Messenger: notice(level) << ... ; everything above the notice level is swallowed
class Messenger
    {
    public:
    Messenger() : m_level(2) { m_null.setstate(std::ios_base::badbit); }
    std::ostream& notice(unsigned int level) { return level <= m_level ? std::cout : m_null; }
    std::ostream& warning() { return std::cerr; }
    std::ostream& error() { return std::cerr; }
    void setNoticeLevel(unsigned int l) { m_level = l; }
    private:
    unsigned int m_level;
    std::ostringstream m_null;
    };

class ExecutionConfiguration
    {
    public:
    explicit ExecutionConfiguration(bool gpu = false, int gpu_id = 0)
        : msg(new Messenger()), m_gpu(gpu), m_gpu_id(gpu_id)
        {
#ifdef ENABLE_HIP
        if (m_gpu)
            {
            cudaError_t e = cudaSetDevice(m_gpu_id);
            if (e != cudaSuccess)
                throw std::runtime_error(std::string("hoomd_shim: cudaSetDevice: ") + cudaGetErrorString(e));
            }
#else
        if (m_gpu)
            throw std::runtime_error("hoomd_shim built without ENABLE_HIP");
#endif
        }
    bool isCUDAEnabled() const { return m_gpu; }
    unsigned int getRank() const { return 0; }
    unsigned int getNRanks() const { return 1; }
    int getGPUId() const { return m_gpu_id; }
    std::shared_ptr<Messenger> msg;
    private:
    bool m_gpu;
    int m_gpu_id;
    };

//! Host/device mirrored array with HOOMD's acquire semantics: asking for the side that is stale
//! copies the whole array across (the cost the reference pays at CavityForceComputeGPU.cc:215-216).
template<class T> class GPUArray
    {
    public:
    GPUArray() : m_n(0), m_dev(nullptr), m_where(0) { }
    GPUArray(size_t n, std::shared_ptr<const ExecutionConfiguration> exec)
        : m_n(n), m_exec(exec), m_host(n), m_dev(nullptr), m_where(0)
        {
        if (n)
            std::memset((void*)m_host.data(), 0, sizeof(T) * n);
#ifdef ENABLE_HIP
        if (m_exec && m_exec->isCUDAEnabled() && n)
            {
            if (cudaMalloc((void**)&m_dev, sizeof(T) * n) != cudaSuccess)
                throw std::runtime_error("hoomd_shim: cudaMalloc failed");
            cudaMemset(m_dev, 0, sizeof(T) * n);
            m_where = 2; // both valid
            }
#endif
        }
    ~GPUArray() { release(); }
    GPUArray(const GPUArray&) = delete;
    GPUArray& operator=(const GPUArray&) = delete;
    GPUArray(GPUArray&& o) noexcept : GPUArray() { swap(o); }
    GPUArray& operator=(GPUArray&& o) noexcept { swap(o); return *this; }
    void swap(GPUArray& o)
        {
        std::swap(m_n, o.m_n); std::swap(m_exec, o.m_exec); m_host.swap(o.m_host);
        std::swap(m_dev, o.m_dev); std::swap(m_where, o.m_where);
        }
    bool isNull() const { return m_n == 0; }
    size_t getNumElements() const { return m_n; }

    T* acquire(access_location::Enum loc, access_mode::Enum mode) const
        {
        if (loc == access_location::host)
            {
#ifdef ENABLE_HIP
            if (m_dev && m_where == 1 && mode != access_mode::overwrite)
                cudaMemcpy((void*)m_host.data(), m_dev, sizeof(T) * m_n, cudaMemcpyDeviceToHost);
#endif
            if (m_dev)
                m_where = (mode == access_mode::read) ? (m_where == 1 ? 2 : m_where) : 0;
            return const_cast<T*>(m_host.data());
            }
#ifdef ENABLE_HIP
        if (!m_dev)
            throw std::runtime_error("hoomd_shim: device access on a host-only array");
        if (m_where == 0 && mode != access_mode::overwrite)
            cudaMemcpy(m_dev, m_host.data(), sizeof(T) * m_n, cudaMemcpyHostToDevice);
        m_where = (mode == access_mode::read) ? (m_where == 0 ? 2 : m_where) : 1;
        return m_dev;
#else
        throw std::runtime_error("hoomd_shim built without ENABLE_HIP");
#endif
        }
    private:
    void release()
        {
#ifdef ENABLE_HIP
        if (m_dev)
            cudaFree(m_dev);
#endif
        m_dev = nullptr;
        }
    size_t m_n;
    std::shared_ptr<const ExecutionConfiguration> m_exec;
    std::vector<T> m_host;
    T* m_dev;
    mutable int m_where; // 0 host valid, 1 device valid, 2 both
    };
template<class T> using GlobalArray = GPUArray<T>;
template<class T> using GlobalVector = GPUArray<T>;

template<class T> class ArrayHandle
    {
    public:
    ArrayHandle(const GPUArray<T>& a,
                access_location::Enum loc = access_location::host,
                access_mode::Enum mode = access_mode::readwrite)
        : data(a.acquire(loc, mode))
        {
        }
    T* const data;
    };

class BoxDim
    {
    public:
    BoxDim() : m_L(make_scalar3(0, 0, 0)) { }
    BoxDim(Scalar Lx, Scalar Ly, Scalar Lz) : m_L(make_scalar3(Lx, Ly, Lz)) { }
    Scalar3 getL() const { return m_L; }
    private:
    Scalar3 m_L;
    };

//! The part of Nano::Signal<void()> the plugin uses: connect / disconnect a member function of an object; emit() calls
//! the connected slots in the order they were connected.
class Signal
    {
    public:
    template<class T, void (T::*M)()> void connect(T* obj) { m_slots.push_back({obj, &thunk<T, M>}); }
    template<class T, void (T::*M)()> void disconnect(T* obj)
        {
        for (size_t k = 0; k < m_slots.size(); k++)
            if (m_slots[k].obj == obj && m_slots[k].fn == &thunk<T, M>)
                {
                m_slots.erase(m_slots.begin() + (std::ptrdiff_t)k);
                return;
                }
        }
    void emit()
        {
        const std::vector<Slot> slots = m_slots;
        for (const Slot& sl : slots)
            sl.fn(sl.obj);
        }
    private:
    template<class T, void (T::*M)()> static void thunk(void* o) { (static_cast<T*>(o)->*M)(); }
    struct Slot
        {
        void* obj;
        void (*fn)(void*);
        };
    std::vector<Slot> m_slots;
    };

class ParticleData
    {
    public:
    ParticleData(unsigned int N, const BoxDim& box, const std::vector<std::string>& types,
                 std::shared_ptr<ExecutionConfiguration> exec)
        : m_N(N), m_box(box), m_types(types), m_exec(exec), m_pos(N, exec), m_vel(N, exec),
          m_accel(N, exec), m_charge(N, exec), m_image(N, exec), m_tag(N, exec), m_net_force(N, exec)
        {
        ArrayHandle<unsigned int> h_tag(m_tag, access_location::host, access_mode::overwrite);
        for (unsigned int i = 0; i < N; i++)
            h_tag.data[i] = i;
        m_rtag.resize(N);
        for (unsigned int i = 0; i < N; i++)
            m_rtag[i] = i;
        }
    unsigned int getN() const { return m_N; }
    unsigned int getNGlobal() const { return m_N; }
    const BoxDim& getGlobalBox() const { return m_box; }
    const BoxDim& getBox() const { return m_box; }
    void setGlobalBox(const BoxDim& b) { m_box = b; }
    const GPUArray<Scalar4>& getPositions() const { return m_pos; }
    const GPUArray<Scalar4>& getVelocities() const { return m_vel; }
    const GPUArray<Scalar3>& getAccelerations() const { return m_accel; }
    const GPUArray<Scalar>& getCharges() const { return m_charge; }
    const GPUArray<int3>& getImages() const { return m_image; }
    const GPUArray<unsigned int>& getTags() const { return m_tag; }
    //! current index of the particle with tag `tag`
    unsigned int getRTag(unsigned int tag) const { return m_rtag.at(tag); }
    //! emitted after the particle arrays were reordered (HOOMD's particle sorter); slots connect with
    //! getParticleSortSignal().connect<Class, &Class::slot>(this)
    Signal& getParticleSortSignal() { return m_sort_signal; }
    //! shim only, what HOOMD's sorter does: the particle now at index j is the one that was at order[j].  Every array
    //! that is indexed by particle moves with it (net force included); then the signal is emitted, and the groups
    //! rebuild their index lists from it.
    void sortParticles(const std::vector<unsigned int>& order)
        {
        if (order.size() != m_N)
            throw std::runtime_error("hoomd_shim: sortParticles needs one index per particle");
        std::vector<char> seen(m_N, 0);
        for (unsigned int o : order)
            {
            if (o >= m_N || seen[o])
                throw std::runtime_error("hoomd_shim: sortParticles needs a permutation");
            seen[o] = 1;
            }
        permute(m_pos, order);
        permute(m_vel, order);
        permute(m_accel, order);
        permute(m_charge, order);
        permute(m_image, order);
        permute(m_net_force, order);
        permute(m_tag, order);
            {
            ArrayHandle<unsigned int> h_tag(m_tag, access_location::host, access_mode::read);
            for (unsigned int i = 0; i < m_N; i++)
                m_rtag[h_tag.data[i]] = i;
            }
        m_sort_signal.emit();
        }
    //! sum of all ForceCompute arrays, formed by the integrator between step one and step two
    const GPUArray<Scalar4>& getNetForce() const { return m_net_force; }
    unsigned int getNTypes() const { return (unsigned int)m_types.size(); }
    unsigned int getTypeByName(const std::string& name) const
        {
        for (unsigned int i = 0; i < m_types.size(); i++)
            if (m_types[i] == name)
                return i;
        throw std::runtime_error("Type " + name + " not found!");
        }
    std::shared_ptr<ExecutionConfiguration> getExecConf() const { return m_exec; }
    private:
    template<class T> void permute(const GPUArray<T>& a, const std::vector<unsigned int>& order)
        {
        ArrayHandle<T> h(a, access_location::host, access_mode::readwrite);
        const std::vector<T> old(h.data, h.data + m_N);
        for (unsigned int j = 0; j < m_N; j++)
            h.data[j] = old[order[j]];
        }
    unsigned int m_N;
    BoxDim m_box;
    std::vector<std::string> m_types;
    std::shared_ptr<ExecutionConfiguration> m_exec;
    GPUArray<Scalar4> m_pos, m_vel;
    GPUArray<Scalar3> m_accel;
    GPUArray<Scalar> m_charge;
    GPUArray<int3> m_image;
    GPUArray<unsigned int> m_tag;
    GPUArray<Scalar4> m_net_force;
    std::vector<unsigned int> m_rtag;
    Signal m_sort_signal;
    };

class SystemDefinition
    {
    public:
    SystemDefinition(std::shared_ptr<ParticleData> pdata, uint16_t seed = 0)
        : m_pdata(pdata), m_seed(seed)
        {
        }
    std::shared_ptr<ParticleData> getParticleData() const { return m_pdata; }
    uint16_t getSeed() const { return m_seed; }
    void setSeed(uint16_t s) { m_seed = s; }
    bool isDomainDecomposed() const { return false; }
    unsigned int getNDimensions() const { return 3; }
    private:
    std::shared_ptr<ParticleData> m_pdata;
    uint16_t m_seed;
    };

//! ForceCompute: owns m_force (Scalar4[N]) and m_virial (6*pitch); compute(t) -> computeForces(t)
class ForceCompute
    {
    public:
    explicit ForceCompute(std::shared_ptr<SystemDefinition> sysdef)
        : m_sysdef(sysdef), m_pdata(sysdef->getParticleData()), m_exec_conf(m_pdata->getExecConf()),
          m_force(m_pdata->getN(), m_exec_conf), m_virial(6 * (size_t)m_pdata->getN(), m_exec_conf),
          m_virial_pitch(m_pdata->getN())
        {
        }
    virtual ~ForceCompute() { }
    void compute(uint64_t timestep) { computeForces(timestep); }
    const GPUArray<Scalar4>& getForceArray() const { return m_force; }
    const GPUArray<Scalar>& getVirialArray() const { return m_virial; }
    //! sum of the per-particle potential energies (force.w), what hoomd's Force.energy reports
    Scalar calcEnergySum()
        {
        ArrayHandle<Scalar4> h(m_force, access_location::host, access_mode::read);
        Scalar e = 0;
        for (unsigned int i = 0; i < m_pdata->getN(); i++)
            e += h.data[i].w;
        return e;
        }
    protected:
    virtual void computeForces(uint64_t timestep) = 0;
    std::shared_ptr<SystemDefinition> m_sysdef;
    std::shared_ptr<ParticleData> m_pdata;
    std::shared_ptr<ExecutionConfiguration> m_exec_conf;
    GPUArray<Scalar4> m_force;
    GPUArray<Scalar> m_virial;
    size_t m_virial_pitch;
    };

//! Autotuner placeholder (the reference constructs one and never uses it, GPU.cc:69-75)
template<size_t n> class Autotuner
    {
    public:
    Autotuner(const std::vector<std::vector<unsigned int>>&, std::shared_ptr<const ExecutionConfiguration>,
              const std::string&, unsigned int = 5) { }
    };

class Variant
    {
    public:
    virtual ~Variant() { }
    virtual Scalar operator()(uint64_t timestep) = 0;
    };
class VariantConstant : public Variant
    {
    public:
    explicit VariantConstant(Scalar v) : m_v(v) { }
    Scalar operator()(uint64_t) override { return m_v; }
    void setValue(Scalar v) { m_v = v; }
    Scalar getValue() const { return m_v; }
    private:
    Scalar m_v;
    };

//! ParticleGroup: a set of particle tags and its index list into the particle arrays.  The shim's particles start with
//! tag == index, so the list is the members as given until the first sort; after a sort it is rebuilt in ascending
//! index order (HOOMD rebuilds it on its sort signal).
class ParticleGroup
    {
    public:
    ParticleGroup(std::shared_ptr<SystemDefinition> sysdef, const std::vector<unsigned int>& members)
        : m_sysdef(sysdef), m_members(members), m_index(members),
          m_idx(members.size(), sysdef->getParticleData()->getExecConf()), m_tdof(0), m_rdof(0)
        {
        ArrayHandle<unsigned int> h(m_idx, access_location::host, access_mode::overwrite);
        for (size_t i = 0; i < members.size(); i++)
            h.data[i] = members[i];
        m_sysdef->getParticleData()->getParticleSortSignal().connect<ParticleGroup, &ParticleGroup::slotParticleSort>(this);
        }
    ~ParticleGroup()
        {
        m_sysdef->getParticleData()->getParticleSortSignal().disconnect<ParticleGroup, &ParticleGroup::slotParticleSort>(this);
        }
    ParticleGroup(const ParticleGroup&) = delete;
    ParticleGroup& operator=(const ParticleGroup&) = delete;
    unsigned int getNumMembers() const { return (unsigned int)m_members.size(); }
    unsigned int getNumMembersGlobal() const { return (unsigned int)m_members.size(); }
    unsigned int getMemberTag(unsigned int i) const { return m_members[i]; }
    unsigned int getMemberIndex(unsigned int i) const { return m_index[i]; }
    const GPUArray<unsigned int>& getIndexArray() const { return m_idx; }
    //! true when the members are exactly first, first+1, ... (lets kernels skip the gather)
    bool isContiguous(unsigned int& first) const
        {
        first = m_index.empty() ? 0 : m_index[0];
        for (size_t i = 0; i < m_index.size(); i++)
            if (m_index[i] != first + i)
                return false;
        return true;
        }
    void slotParticleSort()
        {
        auto pdata = m_sysdef->getParticleData();
        for (size_t i = 0; i < m_members.size(); i++)
            m_index[i] = pdata->getRTag(m_members[i]);
        std::sort(m_index.begin(), m_index.end());
        ArrayHandle<unsigned int> h(m_idx, access_location::host, access_mode::overwrite);
        for (size_t i = 0; i < m_index.size(); i++)
            h.data[i] = m_index[i];
        }
    Scalar getTranslationalDOF() const { return m_tdof; }
    Scalar getRotationalDOF() const { return m_rdof; }
    void setTranslationalDOF(Scalar d) { m_tdof = d; }
    void setRotationalDOF(Scalar d) { m_rdof = d; }
    private:
    std::shared_ptr<SystemDefinition> m_sysdef;
    std::vector<unsigned int> m_members; // tags
    std::vector<unsigned int> m_index;   // their current indices (the host copy of m_idx)
    GPUArray<unsigned int> m_idx;
    Scalar m_tdof, m_rdof;
    };

//! RNG shim.  HOOMD's Philox-based RandomGenerator and its Normal/Gamma samplers are upstream
//! code that is not in the reference tree; the shim makes the draws an INJECTED input so that the
//! reference's arithmetic given the draws is what gets pinned (SURVEY.md section 8c).
struct RNGIdentifier
    {
    enum Enum { BussiThermostat = 0x6a1, MTTKThermostat = 0x6a2 };
    };
struct Seed
    {
    Seed(int id, uint64_t timestep, uint16_t seed) : id(id), timestep(timestep), seed(seed) { }
    int id; uint64_t timestep; uint16_t seed;
    };
struct Counter
    {
    Counter(unsigned int a = 0, unsigned int b = 0, unsigned int c = 0) : a(a) { (void)b; (void)c; }
    unsigned int a;
    };
class RandomGenerator
    {
    public:
    RandomGenerator(const Seed& s, const Counter& c = Counter()) : seed(s), counter(c) { }
    RandomGenerator(const Seed& s, unsigned int instance) : seed(s), counter(instance) { }
    //! draws are consumed in call order from this process-wide queue
    static std::deque<double>& injected()
        {
        static std::deque<double> q;
        return q;
        }
    double next()
        {
        if (injected().empty())
            throw std::runtime_error("hoomd_shim RandomGenerator: no injected draw left");
        double v = injected().front();
        injected().pop_front();
        return v;
        }
    Seed seed;
    Counter counter;
    };
template<class Real> class NormalDistribution
    {
    public:
    explicit NormalDistribution(Real sigma = 1, Real mu = 0) : m_sigma(sigma), m_mu(mu) { }
    Real operator()(RandomGenerator& rng) { return Real(rng.next()) * m_sigma + m_mu; }
    private:
    Real m_sigma, m_mu;
    };
template<class Real> class GammaDistribution
    {
    public:
    GammaDistribution(Real alpha, Real b) : m_alpha(alpha), m_b(b) { }
    //! the injected value is the Gamma(alpha, 1) variate itself
    Real operator()(RandomGenerator& rng) { return Real(rng.next()) * m_b; }
    private:
    Real m_alpha, m_b;
    };

namespace md
    {
//! ComputeThermo: KE = 1/2 sum m|v|^2 over a group (host loop; index-ascending over the group)
class ComputeThermo
    {
    public:
    ComputeThermo(std::shared_ptr<SystemDefinition> sysdef, std::shared_ptr<ParticleGroup> group)
        : m_sysdef(sysdef), m_group(group), m_ke(0)
        {
        }
    virtual ~ComputeThermo() { }
    virtual void compute(uint64_t)
        {
        auto pdata = m_sysdef->getParticleData();
        ArrayHandle<Scalar4> h_vel(pdata->getVelocities(), access_location::host, access_mode::read);
        double ke = 0;
        for (unsigned int j = 0; j < m_group->getNumMembers(); j++)
            {
            const Scalar4 v = h_vel.data[m_group->getMemberIndex(j)];
            ke += v.w * (v.x * v.x + v.y * v.y + v.z * v.z);
            }
        m_ke = 0.5 * ke;
        }
    Scalar getTranslationalDOF() const { return m_group->getTranslationalDOF(); }
    Scalar getRotationalDOF() const { return m_group->getRotationalDOF(); }
    Scalar getTranslationalKineticEnergy() const { return m_ke; }
    //! rotational kinetic energy: HOOMD forms it from angular momenta and moments of inertia (upstream code);
    //! the shim makes it an injected input, like the random draws
    Scalar getRotationalKineticEnergy() const { return m_rke; }
    void setRotationalKineticEnergy(Scalar rke) { m_rke = rke; }
    Scalar getTranslationalTemperature() const
        {
        return getTranslationalDOF() > 0 ? 2.0 * m_ke / getTranslationalDOF() : 0.0;
        }
    Scalar getRotationalTemperature() const { return 0; }
    std::shared_ptr<ParticleGroup> getGroup() const { return m_group; }
    protected:
    std::shared_ptr<SystemDefinition> m_sysdef;
    std::shared_ptr<ParticleGroup> m_group;
    Scalar m_ke;
    Scalar m_rke = 0;
    };
    } // namespace md

    } // namespace hoomd

#endif
