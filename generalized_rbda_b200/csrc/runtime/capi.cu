// Implementation of the C ABI declared in include/grbda_cuda.h.
// Host logic only: model construction / validation, kernel lookup, launches, pinned-memory
// pipelining for host buffers. All per-state arithmetic happens in the generated sm_100a kernels;
// there is deliberately no CPU evaluation path.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <memory>
#include <mutex>
#include <sched.h>
#include <sstream>
#include <string>
#include <sys/syscall.h>
#include <unistd.h>
#include "../../../include/grbda_cuda.h"
#include "../compiler/compile.h"
#include "../host/robots.h"
#include "../host/schedule.h"
#include "jit.h"
#include "registry.h"
#include "support_kernels.cuh"

using namespace grbda;
using grbda_runtime::ModelKernels;

struct grbda_model
{
    ClusterTreeModel model;
    uint64_t hash = 0;
    int device = -1;
    const ModelKernels *kernels = nullptr;         // ahead-of-time kernels (build.py MODELS), or
    std::unique_ptr<grbda_runtime::JitModel> jit;  // kernels compiled at run time (runtime/jit.h)
    // external-force programs for a caller-chosen body set (grbda_cuda_set_external_force_bodies): always
    // compiled at run time, also for models whose other kernels were built ahead of time
    mutable std::unique_ptr<grbda_runtime::JitModel> jit_ext;
    mutable std::mutex jit_ext_mutex;
    bool hasKernels() const { return kernels || jit; }
    // host-buffer pipeline (grbda_cuda_dynamics_host_f64)
    std::mutex host_mutex;
    static constexpr int NSTREAM = 3;
    cudaStream_t streams[NSTREAM] = {nullptr, nullptr, nullptr};
    double *dev_buf[NSTREAM] = {nullptr, nullptr, nullptr};
    double *pin_buf[NSTREAM] = {nullptr, nullptr, nullptr}; // pinned staging for pageable caller buffers
    int64_t dev_capacity = 0; // states per stream buffer
    // per-stream scratch of the kernels (tile flags of the sin/cos range decision). Launches on one
    // stream are ordered, so they can share a buffer; different streams get different buffers.
    struct Scratch
    {
        unsigned char *ptr = nullptr;
        size_t bytes = 0;
    };
    mutable std::mutex scratch_mutex;
    mutable std::string scratch_error;
    mutable std::map<std::pair<cudaStream_t, int>, Scratch> scratch;
    // slot 0: tile flags of a launch; slot 1: intermediate generalized forces of the *_ext entry points;
    // slot 2: accelerations of grbda_cuda_step_f64; slot 3: packed inputs of the vector-Jacobian products;
    // slot 4: the external-force contribution to q_bar of the *_ext_vjp entry points; slot 5: the integration part of
    // grbda_cuda_step_vjp_f64 (q_bar, yd_bar) and its ydd_bar
    unsigned char *scratchFor(cudaStream_t stream, size_t bytes, int slot = 0) const
    {
        std::lock_guard<std::mutex> lock(scratch_mutex);
        Scratch &sc = scratch[{stream, slot}];
        if (sc.bytes < bytes)
        {
            if (sc.ptr)
            {
                cudaStreamSynchronize(stream); // earlier launches on this stream may still use it
                cudaFree(sc.ptr);
            }
            sc.ptr = nullptr;
            sc.bytes = 0;
            const size_t want = std::max<size_t>(bytes * 2, 1 << 16);
            const cudaError_t e = cudaMalloc((void **)&sc.ptr, want);
            if (e != cudaSuccess)
            {
                scratch_error = cudaGetErrorString(e);
                sc.ptr = nullptr;
                return nullptr;
            }
            sc.bytes = want;
        }
        return sc.ptr;
    }
};

namespace
{
    thread_local std::string g_error;
    std::atomic<int64_t> g_launches{0};

    grbda_status fail(grbda_status code, const std::string &msg)
    {
        g_error = msg;
        return code;
    }
    grbda_status cudaFail(cudaError_t e, const char *what)
    {
        return fail(e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? GRBDA_ERR_NO_DEVICE : GRBDA_ERR_CUDA,
                    std::string(what) + ": " + cudaGetErrorString(e));
    }

    int kernelVariant()
    {
        const char *v = std::getenv("GRBDA_KERNEL_VARIANT");
        const int k = v ? std::atoi(v) : 0;
        return k >= 0 && k < grbda_runtime::KERNEL_VARIANTS ? k : 0;
    }

    std::string urdfDirectory()
    {
        if (const char *d = std::getenv("GRBDA_URDF_DIR"))
            return d;
#ifdef GRBDA_DEFAULT_URDF_DIR
        return GRBDA_DEFAULT_URDF_DIR;
#else
        return "robot-models";
#endif
    }

    grbda_status finishCreate(ClusterTreeModel &&m, int device, grbda_model **out)
    {
        grbda_model *h = new grbda_model();
        h->model = std::move(m);
        h->hash = modelHash(h->model);
        h->device = device;
        const int jit_mode = grbda_runtime::jitMode();
        h->kernels = jit_mode == 2 ? nullptr : grbda_runtime::findModelKernels(h->hash);
        if (device >= 0)
        {
            int count = 0;
            cudaError_t e = cudaGetDeviceCount(&count);
            if (e != cudaSuccess || device >= count)
            {
                delete h;
                return e != cudaSuccess ? cudaFail(e, "cudaGetDeviceCount")
                                        : fail(GRBDA_ERR_NO_DEVICE, "device index out of range");
            }
            if (!h->kernels)
            {
                if (jit_mode == 0)
                {
                    char buf[256];
                    std::snprintf(buf, sizeof(buf),
                                  "no sm_100a kernels were compiled ahead of time for this model (hash %016llx) and "
                                  "run-time compilation is disabled (GRBDA_JIT=0)",
                                  (unsigned long long)h->hash);
                    delete h;
                    return fail(GRBDA_ERR_NOT_COMPILED, buf);
                }
                // kernels are compiled by NVRTC when an entry point is first used (or grbda_cuda_model_prepare)
                h->jit.reset(new grbda_runtime::JitModel());
            }
        }
        *out = h;
        return GRBDA_OK;
    }

    template <typename F>
    grbda_status guarded(F f)
    {
        try
        {
            return f();
        }
        catch (const std::exception &e)
        {
            return fail(GRBDA_ERR_INVALID_MODEL, e.what());
        }
    }

    // RAII: make the model's device current for the duration of a call, restore the caller's afterwards
    struct DeviceScope
    {
        int previous = -1;
        cudaError_t error = cudaSuccess;
        explicit DeviceScope(int device)
        {
            error = cudaGetDevice(&previous);
            if (error == cudaSuccess && previous != device)
                error = cudaSetDevice(device);
            else
                previous = -1;
        }
        ~DeviceScope()
        {
            if (previous >= 0)
                cudaSetDevice(previous);
        }
    };

    // sizes of an entry point whatever the kernel source; false: the entry point does not exist for this model
    bool entrySizes(const grbda_model *m, int algo, bool f32, int n_in[3], int n_out[3])
    {
        if (m->kernels)
        {
            const grbda_runtime::AlgoKernels &ak = m->kernels->algo[algo];
            std::memcpy(n_in, ak.n_in, sizeof(ak.n_in));
            std::memcpy(n_out, ak.n_out, sizeof(ak.n_out));
            return (f32 ? ak.f32[0] : ak.f64[0]) != nullptr;
        }
        compiler::algoSizes(m->model, algo, n_in, n_out);
        return n_out[0] > 0;
    }
    bool validEntry(int algo) { return algo >= 0 && algo < compiler::PROGRAM_COUNT && algo != compiler::PROGRAM_FD_LTL; }

    // kernels compiled at run time for every model (programs that depend on caller-chosen sets, reverse mode)
    void ensureExtJit(const grbda_model *m)
    {
        std::lock_guard<std::mutex> lock(m->jit_ext_mutex);
        if (!m->jit_ext)
            m->jit_ext.reset(new grbda_runtime::JitModel());
    }

    grbda_status launchAlgo(const grbda_model *m, int algo, bool f32, const void *in0, const void *in1,
                            const void *in2, void *out0, void *out1, void *out2, int64_t batch, void *stream)
    {
        if (!m)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "null model");
        if (m->device < 0 || !m->hasKernels())
            return fail(GRBDA_ERR_NO_DEVICE, "model was created without a CUDA device (host-only handle)");
        if (batch < 0)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "negative batch");
        DeviceScope scope(m->device);
        if (scope.error != cudaSuccess)
            return cudaFail(scope.error, "cudaSetDevice");
        int n_in[3], n_out[3];
        grbda_runtime::LaunchFn fn = nullptr;
        const grbda_runtime::JitKernel *jk = nullptr;
        // programs that depend on caller-chosen sets (force bodies, contact points) are always run-time compiled
        const bool runtime_only = algo >= compiler::ALGO_CONTACT_KIN;
        if (runtime_only)
        {
            if (grbda_runtime::jitMode() == 0)
                return fail(GRBDA_ERR_NOT_COMPILED, "operational-space programs need run-time compilation (GRBDA_JIT=0)");
            ensureExtJit(m);
        }
        const bool custom_forces = runtime_only || (m->jit_ext && !m->model.externalForceBodies().empty() &&
                                                    (algo == compiler::ALGO_GFA || algo == compiler::ALGO_GFS));
        if (m->kernels && !custom_forces)
        {
            const grbda_runtime::AlgoKernels &ak = m->kernels->algo[algo];
            entrySizes(m, algo, f32, n_in, n_out);
            const char *vs = std::getenv("GRBDA_KERNEL_VARIANT");
            const int v = kernelVariant();
            fn = f32 ? ak.f32[v] : ak.f64[v];
            if (!fn && !vs)
                fn = f32 ? ak.f32[0] : ak.f64[0];
            if (!fn)
                return fail(GRBDA_ERR_NOT_COMPILED, std::string("kernel '") + compiler::algoName(algo) +
                                                        (f32 ? "' (f32)" : "' (f64)") + (vs ? " variant " + std::string(vs) : std::string()) +
                                                        " was not compiled for this model");
        }
        else
        {
            std::string err;
            grbda_runtime::JitModel &jm = custom_forces ? *m->jit_ext : *m->jit;
            if (!grbda_runtime::jitPrepare(jm, m->model, m->hash, m->device, algo, f32, err))
                return fail(GRBDA_ERR_NOT_COMPILED, std::string("kernel '") + compiler::algoName(algo) + "': " + err);
            jk = &jm.algo[algo][f32 ? 1 : 0];
            std::memcpy(n_in, jk->n_in, sizeof(jk->n_in));
            std::memcpy(n_out, jk->n_out, sizeof(jk->n_out));
        }
        if (batch == 0)
            return GRBDA_OK;
        const void *ins[3] = {in0, in1, in2};
        void *outs[3] = {out0, out1, out2};
        for (int i = 0; i < 3; i++)
        {
            if (n_in[i] && !ins[i])
                return fail(GRBDA_ERR_INVALID_ARGUMENT, "null input pointer");
            if (n_out[i] && !outs[i])
                return fail(GRBDA_ERR_INVALID_ARGUMENT, "null output pointer");
            // large outputs (FK p/R/v, H, J, ...) are written with 256-bit (FP32: 128-bit) stores of whole sectors
            if (grbda_kernels::shapeLargeOutput(i, n_out[i]) && ((uintptr_t)outs[i] & (f32 ? 15 : 31)))
                return fail(GRBDA_ERR_INVALID_ARGUMENT, f32 ? "large output arrays must be 16-byte aligned"
                                                            : "large output arrays must be 32-byte aligned");
        }
        grbda_kernels::LaunchArgs a;
        for (int i = 0; i < 3; i++)
        {
            a.in[i] = ins[i];
            a.out[i] = outs[i];
        }
        a.batch = batch;
        a.stream = (cudaStream_t)stream;
        a.flags_bytes = (size_t)((batch + 31) / 32);
        a.flags = m->scratchFor(a.stream, a.flags_bytes);
        if (!a.flags)
            return fail(GRBDA_ERR_CUDA, "cannot allocate the kernel scratch buffer: " + m->scratch_error);
        int launched = 0;
        a.launched = &launched;
        cudaError_t e = jk ? grbda_runtime::jitLaunch(*jk, f32, a) : fn(a);
        if (e != cudaSuccess)
            return cudaFail(e, "kernel launch");
        g_launches += launched ? launched : 1;
        return GRBDA_OK;
    }
} // namespace

extern "C"
{
    const char *grbda_cuda_last_error_string(void) { return g_error.c_str(); }
    const char *grbda_cuda_version(void) { return "grbda_cuda 0.1 (sm_100a)"; }

    grbda_status grbda_cuda_model_create(const grbda_schedule *schedule, int device, grbda_model **out)
    {
        if (!schedule || !out)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "null argument");
        return guarded([&] { return finishCreate(fromSchedule(*schedule), device, out); });
    }
    grbda_status grbda_cuda_model_create_from_urdf(const char *urdf_path, int device, grbda_model **out)
    {
        if (!urdf_path || !out)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "null argument");
        return guarded([&] { return finishCreate(ClusterTreeModel(std::string(urdf_path)), device, out); });
    }
    grbda_status grbda_cuda_model_create_from_urdfs(const char *const *urdf_paths, int num_paths, int device, grbda_model **out)
    {
        if (!urdf_paths || num_paths <= 0 || !out)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "null argument");
        for (int i = 0; i < num_paths; i++)
            if (!urdf_paths[i])
                return fail(GRBDA_ERR_INVALID_ARGUMENT, "null path");
        return guarded([&] {
            return finishCreate(ClusterTreeModel(std::vector<std::string>(urdf_paths, urdf_paths + num_paths)), device, out);
        });
    }
    grbda_status grbda_cuda_describe_urdf(const char *const *urdf_paths, int num_paths, char *json, int64_t capacity,
                                          int64_t *needed)
    {
        if (!urdf_paths || num_paths <= 0)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "null argument");
        return guarded([&] {
            const std::string text = ClusterTreeModel::describeURDF(std::vector<std::string>(urdf_paths, urdf_paths + num_paths));
            if (needed)
                *needed = (int64_t)text.size() + 1;
            if (json && capacity > 0)
            {
                const size_t n = std::min((size_t)capacity - 1, text.size());
                std::memcpy(json, text.data(), n);
                json[n] = 0;
            }
            return GRBDA_OK;
        });
    }
    grbda_status grbda_cuda_model_create_from_robot(const char *name, int device, grbda_model **out)
    {
        if (!name || !out)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "null argument");
        return guarded([&] { return finishCreate(buildRobotByName(name, urdfDirectory()), device, out); });
    }
    grbda_status grbda_cuda_model_destroy(grbda_model *m)
    {
        if (!m)
            return GRBDA_OK;
        for (int i = 0; i < grbda_model::NSTREAM; i++)
        {
            if (m->dev_buf[i])
                cudaFree(m->dev_buf[i]);
            if (m->pin_buf[i])
                cudaFreeHost(m->pin_buf[i]);
            if (m->streams[i])
                cudaStreamDestroy(m->streams[i]);
        }
        for (auto &kv : m->scratch)
            if (kv.second.ptr)
                cudaFree(kv.second.ptr);
        if (m->jit)
            grbda_runtime::jitRelease(*m->jit);
        if (m->jit_ext)
            grbda_runtime::jitRelease(*m->jit_ext);
        delete m;
        return GRBDA_OK;
    }

    int grbda_cuda_num_positions(const grbda_model *m) { return m ? m->model.getNumPositions() : -1; }
    int grbda_cuda_num_degrees_of_freedom(const grbda_model *m) { return m ? m->model.getNumDegreesOfFreedom() : -1; }
    int grbda_cuda_num_bodies(const grbda_model *m) { return m ? m->model.getNumBodies() : -1; }
    int grbda_cuda_num_clusters(const grbda_model *m) { return m ? m->model.getNumClusters() : -1; }
    uint64_t grbda_cuda_model_hash(const grbda_model *m) { return m ? m->hash : 0; }

    grbda_status grbda_cuda_cluster_info(const grbda_model *m, int cluster, int32_t *info8, char *type_name64)
    {
        if (!m || cluster < 0 || cluster >= m->model.getNumClusters() || !info8)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad cluster index");
        const ClusterTreeNode &c = m->model.clusters()[cluster];
        info8[0] = c.parent_index_;
        info8[1] = c.joint_.num_bodies;
        info8[2] = c.num_positions_;
        info8[3] = c.num_velocities_;
        info8[4] = c.position_index_;
        info8[5] = c.velocity_index_;
        info8[6] = (int32_t)c.joint_.type;
        info8[7] = c.first_body_;
        if (type_name64)
            std::snprintf(type_name64, 64, "%s", c.joint_.joint_type_name.c_str());
        return GRBDA_OK;
    }
    grbda_status grbda_cuda_body_info(const grbda_model *m, int body, char *name64, int32_t *info4,
                                      double *E9, double *r3, double *I36)
    {
        if (!m || body < 0 || body >= m->model.getNumBodies())
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad body index");
        const Body &b = m->model.bodies()[body];
        const int ci = m->model.getIndexOfClusterContainingBody(body);
        if (name64)
            std::snprintf(name64, 64, "%s", b.name_.c_str());
        if (info4)
        {
            info4[0] = b.parent_index_;
            info4[1] = ci;
            info4[2] = b.sub_index_within_cluster_;
            info4[3] = (int32_t)m->model.clusters()[ci].joint_.axes[b.sub_index_within_cluster_];
        }
        if (E9)
            std::memcpy(E9, b.Xtree_.E.data(), 72);
        if (r3)
            std::memcpy(r3, b.Xtree_.r.data(), 24);
        if (I36)
            std::memcpy(I36, b.inertia_.getMatrix().data(), 288);
        return GRBDA_OK;
    }
    grbda_status grbda_cuda_cluster_G(const grbda_model *m, int cluster, double *G)
    {
        if (!m || cluster < 0 || cluster >= m->model.getNumClusters() || !G)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad cluster index");
        const ClusterDesc &d = m->model.clusters()[cluster].joint_;
        if (d.type != ClusterType::Explicit)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "cluster has no constant G");
        std::memcpy(G, d.G.data(), d.G.size() * 8);
        return GRBDA_OK;
    }
    grbda_status grbda_cuda_model_gravity(const grbda_model *m, double *gravity3)
    {
        if (!m || !gravity3)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad arguments");
        for (int i = 0; i < 3; i++)
            gravity3[i] = m->model.getGravity()[i];
        return GRBDA_OK;
    }
    grbda_status grbda_cuda_cluster_phi(const grbda_model *m, int cluster, grbda_phi_op *ops, int32_t *outputs,
                                        uint8_t *independent, int32_t *sizes2)
    {
        if (!m || cluster < 0 || cluster >= m->model.getNumClusters() || !sizes2)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad cluster index");
        const ClusterDesc &d = m->model.clusters()[cluster].joint_;
        if (d.type != ClusterType::Implicit)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "cluster has no implicit constraint");
        sizes2[0] = (int32_t)d.phi.ops.size();
        sizes2[1] = (int32_t)d.phi.outputs.size();
        if (ops)
            for (size_t i = 0; i < d.phi.ops.size(); i++)
                ops[i] = grbda_phi_op{d.phi.ops[i].op, d.phi.ops[i].a, d.phi.ops[i].b, d.phi.ops[i].val};
        if (outputs)
            for (size_t i = 0; i < d.phi.outputs.size(); i++)
                outputs[i] = d.phi.outputs[i];
        if (independent)
            for (size_t i = 0; i < d.independent.size(); i++)
                independent[i] = d.independent[i];
        return GRBDA_OK;
    }
    grbda_status grbda_cuda_dump_program(const grbda_model *m, int algo, const char *path, int64_t *counts8)
    {
        if (!m || algo < 0 || algo >= compiler::PROGRAM_COUNT)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad arguments");
        return guarded([&]
                       {
            const compiler::CompiledAlgo c = compiler::compileAlgo(m->model, algo, false);
            if (path)
                compiler::writeTape(c, path);
            if (counts8)
            {
                const compiler::ProgramStats &s = c.stats;
                const int64_t v[8] = {s.n_nodes, s.n_add, s.n_mul, s.n_div, s.n_sqrt, s.n_sin, s.n_cos, s.n_fusable};
                std::memcpy(counts8, v, sizeof(v));
            }
            return (grbda_status)GRBDA_OK; });
    }

    grbda_status grbda_cuda_emit_source(const grbda_model *m, int program, int park, const char *path)
    {
        if (!m || !path || program < 0 || program >= compiler::PROGRAM_COUNT)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad arguments");
        return guarded([&]
                       {
            compiler::ConstTable consts;
            const compiler::CompiledAlgo c = compiler::compileAlgo(m->model, program, true, 0, &consts, 16, park != 0, true, park > 1 ? park - 1 : 0);
            std::ofstream f(path);
            if (!f)
                return fail(GRBDA_ERR_IO, std::string("cannot write ") + path);
            f << consts.definition("kc_table");
            compiler::emitBodyStruct(f, "Body", c);
            return (grbda_status)GRBDA_OK; });
    }

    grbda_status grbda_cuda_kernel_counts(const grbda_model *m, int algo, int64_t *counts8)
    {
        if (!m || !counts8 || algo < 0 || algo >= compiler::ALGO_COUNT)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad arguments");
        if (m->jit)
        {
            std::string err;
            if (!grbda_runtime::jitPrepare(*m->jit, m->model, m->hash, m->device, algo, false, err))
                return fail(GRBDA_ERR_NOT_COMPILED, err);
            std::memcpy(counts8, m->jit->algo[algo][0].counts, 8 * sizeof(int64_t));
            return GRBDA_OK;
        }
        if (!m->kernels || !m->kernels->algo[algo].f64[0])
            return fail(GRBDA_ERR_NOT_COMPILED, "no compiled kernel for this model / algorithm");
        std::memcpy(counts8, m->kernels->algo[algo].counts, 8 * sizeof(int64_t));
        return GRBDA_OK;
    }

    // ---- device-pointer hot path -------------------------------------------------------------------
    grbda_status grbda_cuda_inverse_dynamics_f64(const grbda_model *m, const double *q, const double *yd,
                                                 const double *ydd, double *tau, int64_t batch, void *stream)
    {
        return launchAlgo(m, compiler::ALGO_ID, false, q, yd, ydd, tau, nullptr, nullptr, batch, stream);
    }
    grbda_status grbda_cuda_inverse_dynamics_f32(const grbda_model *m, const float *q, const float *yd,
                                                 const float *ydd, float *tau, int64_t batch, void *stream)
    {
        return launchAlgo(m, compiler::ALGO_ID, true, q, yd, ydd, tau, nullptr, nullptr, batch, stream);
    }
    grbda_status grbda_cuda_forward_dynamics_f64(const grbda_model *m, const double *q, const double *yd,
                                                 const double *tau, double *ydd, int64_t batch, void *stream)
    {
        return launchAlgo(m, compiler::ALGO_FD, false, q, yd, tau, ydd, nullptr, nullptr, batch, stream);
    }
    // ---- external forces on the terminal links ------------------------------------------------
    grbda_status grbda_cuda_external_force_bodies(const grbda_model *m, int32_t *body_indices, int32_t *count)
    {
        if (!m || !count)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad arguments");
        return guarded([&]
                       {
            const std::vector<int> b = compiler::ModelCompiler::externalForceBodies(m->model);
            *count = (int32_t)b.size();
            if (body_indices)
                for (size_t i = 0; i < b.size(); i++)
                    body_indices[i] = b[i];
            return (grbda_status)GRBDA_OK; });
    }
    grbda_status grbda_cuda_set_external_force_bodies(grbda_model *m, const int32_t *body_indices, int32_t count)
    {
        if (!m || count < 0 || (count > 0 && !body_indices))
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad arguments");
        return guarded([&]
                       {
            // launches that still use the old programs must have finished
            if (m->device >= 0)
            {
                DeviceScope scope(m->device);
                cudaDeviceSynchronize();
            }
            m->model.setExternalForceBodies(std::vector<int>(body_indices, body_indices + count));
            if (m->jit_ext)
                grbda_runtime::jitRelease(*m->jit_ext);
            m->jit_ext.reset();
            if (count > 0 && m->device >= 0)
            {
                if (grbda_runtime::jitMode() == 0 && m->kernels)
                    return fail(GRBDA_ERR_NOT_COMPILED, "a custom external-force body set needs run-time compilation (GRBDA_JIT=0)");
                m->jit_ext.reset(new grbda_runtime::JitModel());
            }
            if (m->jit) // a run-time compiled model: its force programs are rebuilt for the new set
                for (int a : {compiler::ALGO_GFA, compiler::ALGO_GFS})
                    for (int p = 0; p < 2; p++)
                        if (m->jit->algo[a][p].ready || !m->jit->algo[a][p].error.empty())
                        {
                            if (m->jit->algo[a][p].library)
                                cudaLibraryUnload(m->jit->algo[a][p].library);
                            m->jit->algo[a][p] = grbda_runtime::JitKernel();
                        }
            return (grbda_status)GRBDA_OK; });
    }

    grbda_status grbda_cuda_inverse_dynamics_ext_f64(const grbda_model *m, const double *q, const double *yd,
                                                     const double *ydd, const double *f_ext, double *tau,
                                                     int64_t batch, void *stream)
    {
        if (!f_ext)
            return launchAlgo(m, compiler::ALGO_ID, false, q, yd, ydd, tau, nullptr, nullptr, batch, stream);
        if (!m || batch < 0)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad arguments");
        if (batch == 0)
            return GRBDA_OK;
        const size_t bytes = (size_t)batch * m->model.getNumDegreesOfFreedom() * sizeof(double);
        double *tmp = (double *)m->scratchFor((cudaStream_t)stream, bytes, 1);
        if (!tmp)
            return fail(GRBDA_ERR_CUDA, "cannot allocate the intermediate generalized-force buffer: " + m->scratch_error);
        grbda_status st = launchAlgo(m, compiler::ALGO_ID, false, q, yd, ydd, tmp, nullptr, nullptr, batch, stream);
        if (st != GRBDA_OK)
            return st;
        return launchAlgo(m, compiler::ALGO_GFS, false, q, f_ext, tmp, tau, nullptr, nullptr, batch, stream);
    }
    grbda_status grbda_cuda_forward_dynamics_ext_f64(const grbda_model *m, const double *q, const double *yd,
                                                     const double *tau, const double *f_ext, double *ydd,
                                                     int64_t batch, void *stream)
    {
        if (!f_ext)
            return launchAlgo(m, compiler::ALGO_FD, false, q, yd, tau, ydd, nullptr, nullptr, batch, stream);
        if (!m || batch < 0)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad arguments");
        if (batch == 0)
            return GRBDA_OK;
        const size_t bytes = (size_t)batch * m->model.getNumDegreesOfFreedom() * sizeof(double);
        double *tmp = (double *)m->scratchFor((cudaStream_t)stream, bytes, 1);
        if (!tmp)
            return fail(GRBDA_ERR_CUDA, "cannot allocate the intermediate generalized-force buffer: " + m->scratch_error);
        grbda_status st = launchAlgo(m, compiler::ALGO_GFA, false, q, f_ext, tau, tmp, nullptr, nullptr, batch, stream);
        if (st != GRBDA_OK)
            return st;
        return launchAlgo(m, compiler::ALGO_FD, false, q, yd, tmp, ydd, nullptr, nullptr, batch, stream);
    }

    grbda_status grbda_cuda_forward_dynamics_f32(const grbda_model *m, const float *q, const float *yd,
                                                 const float *tau, float *ydd, int64_t batch, void *stream)
    {
        return launchAlgo(m, compiler::ALGO_FD, true, q, yd, tau, ydd, nullptr, nullptr, batch, stream);
    }
    grbda_status grbda_cuda_mass_matrix_f64(const grbda_model *m, const double *q, double *H, int64_t batch,
                                            void *stream)
    {
        return launchAlgo(m, compiler::ALGO_H, false, q, nullptr, nullptr, H, nullptr, nullptr, batch, stream);
    }
    grbda_status grbda_cuda_mass_matrix_f32(const grbda_model *m, const float *q, float *H, int64_t batch,
                                            void *stream)
    {
        return launchAlgo(m, compiler::ALGO_H, true, q, nullptr, nullptr, H, nullptr, nullptr, batch, stream);
    }
    grbda_status grbda_cuda_forward_kinematics_f64(const grbda_model *m, const double *q, const double *yd,
                                                   double *p, double *R, double *v, int64_t batch, void *stream)
    {
        return launchAlgo(m, compiler::ALGO_FK, false, q, yd, nullptr, p, R, v, batch, stream);
    }
    grbda_status grbda_cuda_forward_kinematics_f32(const grbda_model *m, const float *q, const float *yd,
                                                   float *p, float *R, float *v, int64_t batch, void *stream)
    {
        return launchAlgo(m, compiler::ALGO_FK, true, q, yd, nullptr, p, R, v, batch, stream);
    }

    // ---- host-pointer path: chunks pipelined over three streams --------------------------------------
    // mode 0: ID, 1: FD, 2: FD followed by ID of the result (out2 = tau_back).
    // Page-locked caller buffers (cudaHostAlloc / cudaHostRegister / torch pin_memory) are used in place:
    // the copies of one chunk overlap the kernels and copies of the others. Pageable buffers are staged
    // through the handle's own pinned buffers, chunk by chunk, so that the overlap survives (an async copy
    // from pageable memory is synchronous).
    static bool isPinned(const void *p)
    {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, p) != cudaSuccess)
        {
            (void)cudaGetLastError();
            return false;
        }
        return at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged;
    }

    static grbda_status hostPipeline(grbda_model *m, int mode, const double *q, const double *yd,
                                     const double *in3, double *out, double *out2, int64_t batch)
    {
        if (m->device < 0 || !m->hasKernels())
            return fail(GRBDA_ERR_NO_DEVICE, "model was created without a CUDA device (host-only handle)");
        if (batch < 0)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "negative batch");
        std::lock_guard<std::mutex> lock(m->host_mutex);
        DeviceScope scope(m->device);
        cudaError_t e = scope.error;
        if (e != cudaSuccess)
            return cudaFail(e, "cudaSetDevice");
        const int nq = m->model.getNumPositions(), nv = m->model.getNumDegreesOfFreedom();
        const int64_t per_state = nq + 4 * (int64_t)nv; // q, yd, in3, out, out2 (doubles)
        const bool staged = !(isPinned(q) && isPinned(yd) && isPinned(in3) && isPinned(out) && (mode != 2 || isPinned(out2)));
        // measured (tools/e2e_sweep.py, 2^20 Tello states): 16 k -> 57.6, 32 k -> 67.0, 64 k -> 70.7, 128 k -> 72.3,
        // 256 k -> 68.6 M fwd+inv/s; the call is bound by the host link (47 GB/s in, 28 GB/s out, concurrently)
        int64_t chunk = staged ? 1 << 15 : 1 << 17;
        if (const char *c = std::getenv("GRBDA_HOST_CHUNK")) // tuning knob (states per pipelined chunk)
            chunk = std::max<int64_t>(1024, std::atoll(c));
        if (m->dev_capacity != chunk || (staged && !m->pin_buf[0]))
        {
            for (int i = 0; i < grbda_model::NSTREAM; i++)
            {
                if (!m->streams[i] && (e = cudaStreamCreateWithFlags(&m->streams[i], cudaStreamNonBlocking)) != cudaSuccess)
                    return cudaFail(e, "cudaStreamCreate");
                if (m->dev_capacity != chunk)
                {
                    if (m->dev_buf[i])
                        cudaFree(m->dev_buf[i]);
                    m->dev_buf[i] = nullptr;
                    if (m->pin_buf[i])
                        cudaFreeHost(m->pin_buf[i]);
                    m->pin_buf[i] = nullptr;
                    if ((e = cudaMalloc(&m->dev_buf[i], chunk * per_state * sizeof(double))) != cudaSuccess)
                        return cudaFail(e, "cudaMalloc");
                }
                if (staged && !m->pin_buf[i] &&
                    (e = cudaHostAlloc((void **)&m->pin_buf[i], chunk * per_state * sizeof(double), cudaHostAllocDefault)) != cudaSuccess)
                    return cudaFail(e, "cudaHostAlloc");
            }
            m->dev_capacity = chunk;
        }
        // staged mode: results of the chunk a stream worked on last, still to be copied to the caller
        struct Pending
        {
            int64_t b0 = 0, nb = 0;
        } pending[grbda_model::NSTREAM];
        grbda_status rs = GRBDA_OK;
        auto drain = [&](int s) -> cudaError_t
        {
            cudaError_t de = cudaStreamSynchronize(m->streams[s]);
            if (de == cudaSuccess && staged && pending[s].nb)
            {
                const double *pout = m->pin_buf[s] + chunk * (nq + 2 * (int64_t)nv);
                std::memcpy(out + pending[s].b0 * nv, pout, pending[s].nb * nv * 8);
                if (mode == 2)
                    std::memcpy(out2 + pending[s].b0 * nv, pout + chunk * nv, pending[s].nb * nv * 8);
            }
            pending[s].nb = 0;
            return de;
        };
        // Chunk sizes. The first chunk's upload and the last chunk's download overlap with nothing, so the pipeline
        // opens and closes with short chunks (1/8, 1/4, 1/2 of the steady-state size) - uniformly short chunks are
        // slower (tools/e2e_sweep.py). Measured: 14.47 -> 14.37 ms per 2^20 Tello states at 128 k chunks, 15.18 -> 14.66 ms
        // at 256 k: the call sits on the duplex host link (H2D 47 GB/s while D2H runs), not on fill and drain.
        // GRBDA_HOST_RAMP=0: uniform chunks.
        std::vector<int64_t> sizes;
        {
            static const bool ramp = !(std::getenv("GRBDA_HOST_RAMP") && std::getenv("GRBDA_HOST_RAMP")[0] == '0');
            const int64_t edge[3] = {chunk / 8, chunk / 4, chunk / 2};
            const int64_t edges = edge[0] + edge[1] + edge[2];
            int64_t left = batch;
            if (ramp && chunk >= 8192 && batch >= 2 * chunk)
            {
                for (int i = 0; i < 3; i++)
                    sizes.push_back(edge[i]);
                left -= 2 * edges;
            }
            const bool ramped = !sizes.empty();
            for (; left > 0; left -= chunk)
                sizes.push_back(std::min(chunk, left));
            if (ramped)
                for (int i = 2; i >= 0; i--)
                    sizes.push_back(edge[i]);
        }
        int64_t b0 = 0;
        for (size_t k = 0; k < sizes.size() && rs == GRBDA_OK; b0 += sizes[k], k++)
        {
            const int64_t nb = sizes[k];
            const int s = (int)(k % grbda_model::NSTREAM);
            cudaStream_t st = m->streams[s];
            double *dq = m->dev_buf[s], *dyd = dq + chunk * nq, *din = dyd + chunk * nv, *dout = din + chunk * nv,
                   *dout2 = dout + chunk * nv;
            const double *hq = q + b0 * nq, *hyd = yd + b0 * nv, *hin = in3 + b0 * nv;
            double *hout = out + b0 * nv, *hout2 = out2 ? out2 + b0 * nv : nullptr;
            if (staged)
            {
                if ((e = drain(s)) != cudaSuccess) // the stream's pinned buffer is free again
                {
                    rs = cudaFail(e, "cudaStreamSynchronize");
                    break;
                }
                double *pq = m->pin_buf[s], *pyd = pq + chunk * nq, *pin = pyd + chunk * nv, *pout = pin + chunk * nv;
                std::memcpy(pq, hq, nb * nq * 8);
                std::memcpy(pyd, hyd, nb * nv * 8);
                std::memcpy(pin, hin, nb * nv * 8);
                hq = pq, hyd = pyd, hin = pin, hout = pout, hout2 = pout + chunk * nv;
                pending[s].b0 = b0, pending[s].nb = nb;
            }
            if ((e = cudaMemcpyAsync(dq, hq, nb * nq * 8, cudaMemcpyHostToDevice, st)) != cudaSuccess ||
                (e = cudaMemcpyAsync(dyd, hyd, nb * nv * 8, cudaMemcpyHostToDevice, st)) != cudaSuccess ||
                (e = cudaMemcpyAsync(din, hin, nb * nv * 8, cudaMemcpyHostToDevice, st)) != cudaSuccess)
            {
                rs = cudaFail(e, "cudaMemcpyAsync H2D");
                break;
            }
            rs = launchAlgo(m, mode == 0 ? compiler::ALGO_ID : compiler::ALGO_FD, false, dq, dyd, din, dout, nullptr,
                            nullptr, nb, st);
            if (rs != GRBDA_OK)
                break;
            if ((e = cudaMemcpyAsync(hout, dout, nb * nv * 8, cudaMemcpyDeviceToHost, st)) != cudaSuccess)
            {
                rs = cudaFail(e, "cudaMemcpyAsync D2H");
                break;
            }
            if (mode == 2)
            {
                rs = launchAlgo(m, compiler::ALGO_ID, false, dq, dyd, dout, dout2, nullptr, nullptr, nb, st);
                if (rs != GRBDA_OK)
                    break;
                if ((e = cudaMemcpyAsync(hout2, dout2, nb * nv * 8, cudaMemcpyDeviceToHost, st)) != cudaSuccess)
                {
                    rs = cudaFail(e, "cudaMemcpyAsync D2H");
                    break;
                }
            }
        }
        // also on the error paths: no copy on a caller buffer may still be in flight when the call returns
        const std::string first_error = g_error;
        for (int i = 0; i < grbda_model::NSTREAM; i++)
            if (m->streams[i] && (e = drain(i)) != cudaSuccess && rs == GRBDA_OK)
                rs = cudaFail(e, "cudaStreamSynchronize");
        if (rs != GRBDA_OK && !first_error.empty())
            g_error = first_error;
        return rs;
    }

    grbda_status grbda_cuda_dynamics_host_f64(const grbda_model *cm, int algo, const double *q, const double *yd,
                                              const double *in3, double *out, int64_t batch)
    {
        grbda_model *m = const_cast<grbda_model *>(cm);
        if (!m || (algo != 0 && algo != 1) || !q || !yd || !in3 || !out)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad arguments");
        return hostPipeline(m, algo, q, yd, in3, out, nullptr, batch);
    }
    grbda_status grbda_cuda_forward_inverse_host_f64(const grbda_model *cm, const double *q, const double *yd,
                                                     const double *tau, double *ydd, double *tau_back,
                                                     int64_t batch)
    {
        grbda_model *m = const_cast<grbda_model *>(cm);
        if (!m || !q || !yd || !tau || !ydd || !tau_back)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad arguments");
        return hostPipeline(m, 2, q, yd, tau, ydd, tau_back, batch);
    }

    // ---- kernel provenance / run-time compilation ------------------------------------------------------
    grbda_status grbda_cuda_model_prepare(const grbda_model *m, int algo, int f32)
    {
        if (!m || (algo != GRBDA_PROGRAM_INTEGRATE_VJP && !validEntry(algo)))
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad arguments");
        if (m->device < 0 || !m->hasKernels())
            return fail(GRBDA_ERR_NO_DEVICE, "model was created without a CUDA device (host-only handle)");
        if (algo == GRBDA_PROGRAM_INTEGRATE_VJP)
        {
            if (grbda_runtime::jitMode() == 0)
                return fail(GRBDA_ERR_NOT_COMPILED, "the reverse integration step needs run-time compilation (GRBDA_JIT=0)");
            ensureExtJit(m);
            std::string err;
            if (!grbda_runtime::jitPrepareIntegrateVjp(*m->jit_ext, m->model, m->device, err))
                return fail(GRBDA_ERR_NOT_COMPILED, "reverse integration step: " + err);
            return GRBDA_OK;
        }
        if (algo == compiler::ALGO_CONTACT_FD || algo == compiler::ALGO_CONTACT_IMPULSE)
        {
            if (grbda_runtime::jitMode() == 0)
                return fail(GRBDA_ERR_NOT_COMPILED, "rigid-contact programs need run-time compilation (GRBDA_JIT=0)");
            if (f32 || m->model.contactPoints().empty())
                return fail(GRBDA_ERR_INVALID_ARGUMENT, "rigid-contact programs: FP64 and a contact set only");
            ensureExtJit(m);
            std::string err;
            if (!grbda_runtime::jitPrepare(*m->jit_ext, m->model, m->hash, m->device, algo, false, err))
                return fail(GRBDA_ERR_NOT_COMPILED, err);
            return GRBDA_OK;
        }
        if (algo >= compiler::ALGO_CONTACT_KIN)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "operational-space programs are compiled when first used");
        if (m->kernels)
            return (f32 ? m->kernels->algo[algo].f32[0] : m->kernels->algo[algo].f64[0])
                       ? GRBDA_OK
                       : fail(GRBDA_ERR_NOT_COMPILED, "entry point was not compiled ahead of time for this model");
        std::string err;
        if (!grbda_runtime::jitPrepare(*m->jit, m->model, m->hash, m->device, algo, f32 != 0, err))
            return fail(GRBDA_ERR_NOT_COMPILED, err);
        return GRBDA_OK;
    }

    grbda_status grbda_cuda_kernel_info(const grbda_model *m, int algo, int f32, int64_t *info8)
    {
        if (!m || !info8 || !validEntry(algo))
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad arguments");
        std::memset(info8, 0, 8 * sizeof(int64_t));
        if (m->kernels && algo < compiler::ALGO_COUNT)
        {
            info8[0] = 0;
            info8[7] = (f32 ? m->kernels->algo[algo].f32[0] : m->kernels->algo[algo].f64[0]) ? 1 : 0;
            return GRBDA_OK;
        }
        return guarded([&]
                       {
            grbda_runtime::JitKernel local;
            const grbda_runtime::JitKernel *k = &local;
            std::string err;
            if (m->jit && m->jit->algo[algo][f32 ? 1 : 0].ready)
                k = &m->jit->algo[algo][f32 ? 1 : 0];
            else if (m->jit_ext && m->jit_ext->algo[algo][f32 ? 1 : 0].ready)
                k = &m->jit_ext->algo[algo][f32 ? 1 : 0];
            else if (!grbda_runtime::jitDescribe(m->model, algo, f32 != 0, local, err))
                return fail(GRBDA_ERR_NOT_COMPILED, err);
            info8[0] = 1;
            info8[1] = k->shape.block;
            info8[2] = k->shape.min_blocks;
            info8[3] = (int64_t)k->shape.smem_fast;
            info8[4] = k->shape.program;
            info8[5] = (k->shape.park ? 1 : 0) | (k->shape.kind == 'T' ? 2 : 0) | (k->shape.kind == 'D' ? 4 : 0) |
                       (k->from_cache ? 8 : 0);
            info8[6] = (int64_t)(k->compile_seconds * 1000.0);
            info8[7] = k->ready ? 1 : 0;
            return (grbda_status)GRBDA_OK; });
    }

    grbda_status grbda_cuda_jit_compile(const grbda_model *m, int algo, int f32, const char *source_path,
                                        const char *cubin_path)
    {
        if (!m || (algo != -1 && algo != GRBDA_PROGRAM_INTEGRATE_VJP && !validEntry(algo)))
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad arguments");
        return guarded([&]
                       {
            grbda_runtime::JitKernel k;
            std::vector<std::string> names, lowered;
            const std::string src = algo == -1 ? grbda_runtime::jitGenerateSource(m->model, names)
                                    : algo == GRBDA_PROGRAM_INTEGRATE_VJP ? grbda_runtime::jitIntegrateVjpSource(m->model, names)
                                                                          : grbda_runtime::jitSource(m->model, algo, f32 != 0, k, names);
            if (source_path)
            {
                std::ofstream f(source_path);
                if (!f)
                    return fail(GRBDA_ERR_IO, std::string("cannot write ") + source_path);
                f << src;
                for (auto &n : names)
                    f << "// kernel: " << n << "\n";
            }
            if (cubin_path)
            {
                std::vector<char> cubin;
                std::string log;
                if (!grbda_runtime::jitCompile(src, names, cubin, lowered, log))
                    return fail(GRBDA_ERR_NOT_COMPILED, log);
                std::ofstream f(cubin_path, std::ios::binary);
                if (!f)
                    return fail(GRBDA_ERR_IO, std::string("cannot write ") + cubin_path);
                f.write(cubin.data(), (std::streamsize)cubin.size());
            }
            return (grbda_status)GRBDA_OK; });
    }

    // ---- operational space (SURVEY 8 f1) ---------------------------------------------------------------------
    grbda_status grbda_cuda_set_contact_points(grbda_model *m, int32_t count, const int32_t *body_indices,
                                               const double *local_offsets, const uint8_t *is_end_effector)
    {
        if (!m || count < 0 || (count > 0 && (!body_indices || !local_offsets)))
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad arguments");
        return guarded([&]
                       {
            if (m->device >= 0)
            {
                DeviceScope scope(m->device);
                cudaDeviceSynchronize();
            }
            std::vector<ContactPoint> pts;
            for (int i = 0; i < count; i++)
                pts.push_back(ContactPoint{body_indices[i], {local_offsets[3 * i], local_offsets[3 * i + 1], local_offsets[3 * i + 2]},
                                           "contact-" + std::to_string(i), is_end_effector && is_end_effector[i] != 0});
            m->model.setContactPoints(pts);
            std::lock_guard<std::mutex> lock(m->jit_ext_mutex);
            if (m->jit_ext)
                for (int a : {compiler::ALGO_CONTACT_KIN, compiler::ALGO_CONTACT_JAC, compiler::ALGO_TEST_FORCE,
                              compiler::ALGO_OSIM, compiler::ALGO_CONTACT_KIN_VJP, compiler::ALGO_CONTACT_FD,
                              compiler::ALGO_CONTACT_IMPULSE})
                    for (int p = 0; p < 2; p++)
                    {
                        if (m->jit_ext->algo[a][p].library)
                            cudaLibraryUnload(m->jit_ext->algo[a][p].library);
                        m->jit_ext->algo[a][p] = grbda_runtime::JitKernel();
                    }
            return (grbda_status)GRBDA_OK; });
    }
    int grbda_cuda_num_contact_points(const grbda_model *m) { return m ? (int)m->model.contactPoints().size() : -1; }
    int grbda_cuda_num_end_effectors(const grbda_model *m) { return m ? m->model.getNumEndEffectors() : -1; }

    grbda_status grbda_cuda_contact_kinematics_f64(const grbda_model *m, const double *q, const double *yd, double *p,
                                                   double *v, int64_t batch, void *stream)
    {
        if (m && m->model.contactPoints().empty())
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "the model has no contact points (grbda_cuda_set_contact_points)");
        return launchAlgo(m, compiler::ALGO_CONTACT_KIN, false, q, yd, nullptr, p, v, nullptr, batch, stream);
    }
    grbda_status grbda_cuda_contact_jacobians_f64(const grbda_model *m, const double *q, double *J, int64_t batch,
                                                  void *stream)
    {
        if (m && m->model.contactPoints().empty())
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "the model has no contact points (grbda_cuda_set_contact_points)");
        return launchAlgo(m, compiler::ALGO_CONTACT_JAC, false, q, nullptr, nullptr, J, nullptr, nullptr, batch, stream);
    }
    grbda_status grbda_cuda_apply_test_force_f64(const grbda_model *m, const double *q, const double *force,
                                                 double *dstate, double *lambda_inv, int64_t batch, void *stream)
    {
        if (m && m->model.contactPoints().empty())
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "the model has no contact points (grbda_cuda_set_contact_points)");
        return launchAlgo(m, compiler::ALGO_TEST_FORCE, false, q, force, nullptr, dstate, lambda_inv, nullptr, batch, stream);
    }
    grbda_status grbda_cuda_inverse_dynamics_derivatives_f64(const grbda_model *m, const double *q, const double *yd,
                                                             const double *ydd, double *dtau_dq, double *dtau_dyd,
                                                             int64_t batch, void *stream)
    {
        return launchAlgo(m, compiler::ALGO_ID_DERIV, false, q, yd, ydd, dtau_dq, dtau_dyd, nullptr, batch, stream);
    }
    grbda_status grbda_cuda_forward_dynamics_derivatives_f64(const grbda_model *m, const double *q, const double *yd,
                                                             const double *tau, double *dydd_dq, double *dydd_dyd,
                                                             double *dydd_dtau, int64_t batch, void *stream)
    {
        return launchAlgo(m, compiler::ALGO_FD_DERIV, false, q, yd, tau, dydd_dq, dydd_dyd, dydd_dtau, batch, stream);
    }
}

namespace
{
    // Checks shared by the vector-Jacobian product entry points, before any pointer (batch = 0 launches nothing)
    grbda_status vjpCheck(const grbda_model *m, int64_t batch)
    {
        if (!m)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "null model");
        if (m->device < 0 || !m->hasKernels())
            return fail(GRBDA_ERR_NO_DEVICE, "model was created without a CUDA device (host-only handle)");
        if (batch < 0)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "negative batch");
        if (grbda_runtime::jitMode() == 0)
            return fail(GRBDA_ERR_NOT_COMPILED, "vector-Jacobian product programs need run-time compilation (GRBDA_JIT=0)");
        return GRBDA_OK;
    }

    // The kernels of the shells read three input arrays per state: two per-state arrays x [batch][nx] and
    // y [batch][ny] (the third argument and the cotangent, or two cotangents) are packed into [batch][nx + ny]
    // (scratch slot 3) with two pitched device-to-device copies on the caller's stream.
    grbda_status packRows(const grbda_model *m, const double *x, size_t nx, const double *y, size_t ny, int64_t batch,
                          cudaStream_t stream, double *&packed)
    {
        const size_t row = (nx + ny) * sizeof(double);
        packed = (double *)m->scratchFor(stream, (size_t)batch * row, 3);
        if (!packed)
            return fail(GRBDA_ERR_CUDA, "cannot allocate the packed input buffer: " + m->scratch_error);
        cudaError_t e = cudaMemcpy2DAsync(packed, row, x, nx * sizeof(double), nx * sizeof(double), (size_t)batch,
                                          cudaMemcpyDeviceToDevice, stream);
        if (e == cudaSuccess)
            e = cudaMemcpy2DAsync(packed + nx, row, y, ny * sizeof(double), ny * sizeof(double), (size_t)batch,
                                  cudaMemcpyDeviceToDevice, stream);
        if (e != cudaSuccess)
            return cudaFail(e, "packing the vector-Jacobian product inputs");
        return GRBDA_OK;
    }

    grbda_status launchVJP(const grbda_model *m, int algo, const double *q, const double *yd, const double *aux,
                           const double *w, double *q_bar, double *yd_bar, double *aux_bar, int64_t batch, void *stream)
    {
        grbda_status st = vjpCheck(m, batch);
        if (st != GRBDA_OK || batch == 0)
            return st;
        if (!aux || !w)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "null input pointer");
        DeviceScope scope(m->device);
        if (scope.error != cudaSuccess)
            return cudaFail(scope.error, "cudaSetDevice");
        const size_t nv = (size_t)m->model.getNumDegreesOfFreedom();
        double *packed = nullptr;
        if ((st = packRows(m, aux, nv, w, nv, batch, (cudaStream_t)stream, packed)) != GRBDA_OK)
            return st;
        return launchAlgo(m, algo, false, q, yd, packed, q_bar, yd_bar, aux_bar, batch, stream);
    }

    // y0 += x0, y1 += x1 (n0, n1 doubles) in one launch
    grbda_status accumulate(double *y0, const double *x0, int64_t n0, double *y1, const double *x1, int64_t n1,
                            cudaStream_t s)
    {
        const int64_t n = n0 + n1;
        const int grid = (int)std::min<int64_t>((n + 255) / 256, 148 * 8);
        grbda_kernels::accumulateKernel<<<grid, 256, 0, s>>>(y0, x0, n0, y1, x1, n1);
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess)
            return cudaFail(e, "accumulateKernel");
        g_launches++;
        return GRBDA_OK;
    }

    // The dynamics VJP with external forces, composed of the programs that exist (f_ext != NULL):
    //   inverse dynamics, tau = ID(q, yd, ydd) - J^T f: ALGO_ID_VJP with w, then ALGO_GFS_VJP(q, f, w);
    //   forward dynamics, ydd = FD(q, yd, tau'), tau' = tau + J^T f: ALGO_GFA -> tau' (scratch slot 1), ALGO_FD_VJP at
    //   tau' (tau_bar = H^-1 w), then ALGO_GFA_VJP(q, f, tau_bar).
    // The force program writes f_bar and its q contribution (scratch slot 4), which one more launch adds to q_bar.
    grbda_status launchExtVJP(const grbda_model *m, bool forward, const double *q, const double *yd, const double *aux,
                              const double *f_ext, const double *w, double *q_bar, double *yd_bar, double *aux_bar,
                              double *f_bar, int64_t batch, void *stream)
    {
        grbda_status st = vjpCheck(m, batch);
        if (st != GRBDA_OK || batch == 0)
            return st;
        if (!q || !yd || !aux || !w)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "null input pointer");
        if (!q_bar || !yd_bar || !aux_bar || !f_bar)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "null output pointer");
        DeviceScope scope(m->device);
        if (scope.error != cudaSuccess)
            return cudaFail(scope.error, "cudaSetDevice");
        const cudaStream_t s = (cudaStream_t)stream;
        const int64_t nq = m->model.getNumPositions(), nv = m->model.getNumDegreesOfFreedom();
        double *q_gf = (double *)m->scratchFor(s, (size_t)(batch * nq) * sizeof(double), 4);
        if (!q_gf)
            return fail(GRBDA_ERR_CUDA, "cannot allocate the external-force q_bar buffer: " + m->scratch_error);
        if (forward)
        {
            double *tau_eff = (double *)m->scratchFor(s, (size_t)(batch * nv) * sizeof(double), 1);
            if (!tau_eff)
                return fail(GRBDA_ERR_CUDA, "cannot allocate the intermediate generalized-force buffer: " + m->scratch_error);
            if ((st = launchAlgo(m, compiler::ALGO_GFA, false, q, f_ext, aux, tau_eff, nullptr, nullptr, batch, stream)) != GRBDA_OK ||
                (st = launchVJP(m, compiler::ALGO_FD_VJP, q, yd, tau_eff, w, q_bar, yd_bar, aux_bar, batch, stream)) != GRBDA_OK ||
                (st = launchAlgo(m, compiler::ALGO_GFA_VJP, false, q, f_ext, aux_bar, q_gf, f_bar, nullptr, batch, stream)) != GRBDA_OK)
                return st;
        }
        else if ((st = launchVJP(m, compiler::ALGO_ID_VJP, q, yd, aux, w, q_bar, yd_bar, aux_bar, batch, stream)) != GRBDA_OK ||
                 (st = launchAlgo(m, compiler::ALGO_GFS_VJP, false, q, f_ext, w, q_gf, f_bar, nullptr, batch, stream)) != GRBDA_OK)
            return st;
        return accumulate(q_bar, q_gf, batch * nq, nullptr, nullptr, 0, s);
    }

    // The rigid-contact programs (include/grbda_cuda.h): packContactRowsKernel writes input array 2 into scratch slot 3
    // (the packed inputs of the VJPs), then the program runs, both on the caller's stream
    grbda_status launchContact(const grbda_model *m, int algo, const double *q, const double *yd, const double *tau,
                               const uint8_t *active, double restitution, double damping, double *y_out, double *lambda,
                               int64_t batch, void *stream)
    {
        if (!m)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "null model");
        if (m->model.contactPoints().empty())
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "the model has no contact points (grbda_cuda_set_contact_points)");
        if (!std::isfinite(damping) || damping < 0.0)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "the damping must be finite and >= 0");
        if (!(restitution >= 0.0 && restitution <= 1.0))
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "the restitution must lie in [0, 1]");
        if (m->device < 0 || !m->hasKernels())
            return fail(GRBDA_ERR_NO_DEVICE, "model was created without a CUDA device (host-only handle)");
        if (batch < 0)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "negative batch");
        if (grbda_runtime::jitMode() == 0)
            return fail(GRBDA_ERR_NOT_COMPILED, "rigid-contact programs need run-time compilation (GRBDA_JIT=0)");
        if (batch == 0)
            return GRBDA_OK;
        const bool impulse = algo == compiler::ALGO_CONTACT_IMPULSE;
        if (!q || !yd || (!impulse && !tau))
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "null input pointer");
        if (!y_out || !lambda)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "null output pointer");
        DeviceScope scope(m->device);
        if (scope.error != cudaSuccess)
            return cudaFail(scope.error, "cudaSetDevice");
        const cudaStream_t s = (cudaStream_t)stream;
        const int ncp = (int)m->model.contactPoints().size(), nt = impulse ? 0 : m->model.getNumDegreesOfFreedom();
        const int ns = impulse ? 2 : 1;
        const int64_t n = batch * (nt + ncp + ns);
        double *packed = (double *)m->scratchFor(s, (size_t)n * sizeof(double), 3);
        if (!packed)
            return fail(GRBDA_ERR_CUDA, "cannot allocate the packed input buffer: " + m->scratch_error);
        const int grid = (int)std::min<int64_t>((n + 255) / 256, 148 * 8);
        grbda_kernels::packContactRowsKernel<<<grid, 256, 0, s>>>(packed, tau, nt, active, ncp, impulse ? restitution : damping,
                                                                 damping, ns, batch);
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess)
            return cudaFail(e, "packContactRowsKernel");
        g_launches++;
        return launchAlgo(m, algo, false, q, yd, packed, y_out, lambda, nullptr, batch, stream);
    }
} // namespace

extern "C"
{
    grbda_status grbda_cuda_inverse_dynamics_vjp_f64(const grbda_model *m, const double *q, const double *yd,
                                                     const double *ydd, const double *tau_bar, double *q_bar,
                                                     double *yd_bar, double *ydd_bar, int64_t batch, void *stream)
    {
        return launchVJP(m, compiler::ALGO_ID_VJP, q, yd, ydd, tau_bar, q_bar, yd_bar, ydd_bar, batch, stream);
    }
    grbda_status grbda_cuda_forward_dynamics_vjp_f64(const grbda_model *m, const double *q, const double *yd,
                                                     const double *tau, const double *ydd_bar, double *q_bar,
                                                     double *yd_bar, double *tau_bar, int64_t batch, void *stream)
    {
        return launchVJP(m, compiler::ALGO_FD_VJP, q, yd, tau, ydd_bar, q_bar, yd_bar, tau_bar, batch, stream);
    }
    grbda_status grbda_cuda_inverse_dynamics_ext_vjp_f64(const grbda_model *m, const double *q, const double *yd,
                                                         const double *ydd, const double *f_ext, const double *tau_bar,
                                                         double *q_bar, double *yd_bar, double *ydd_bar, double *f_bar,
                                                         int64_t batch, void *stream)
    {
        if (!f_ext)
            return launchVJP(m, compiler::ALGO_ID_VJP, q, yd, ydd, tau_bar, q_bar, yd_bar, ydd_bar, batch, stream);
        return launchExtVJP(m, false, q, yd, ydd, f_ext, tau_bar, q_bar, yd_bar, ydd_bar, f_bar, batch, stream);
    }
    grbda_status grbda_cuda_forward_dynamics_ext_vjp_f64(const grbda_model *m, const double *q, const double *yd,
                                                         const double *tau, const double *f_ext, const double *ydd_bar,
                                                         double *q_bar, double *yd_bar, double *tau_bar, double *f_bar,
                                                         int64_t batch, void *stream)
    {
        if (!f_ext)
            return launchVJP(m, compiler::ALGO_FD_VJP, q, yd, tau, ydd_bar, q_bar, yd_bar, tau_bar, batch, stream);
        return launchExtVJP(m, true, q, yd, tau, f_ext, ydd_bar, q_bar, yd_bar, tau_bar, f_bar, batch, stream);
    }
    grbda_status grbda_cuda_contact_kinematics_vjp_f64(const grbda_model *m, const double *q, const double *yd,
                                                       const double *p_bar, const double *v_bar, double *q_bar,
                                                       double *yd_bar, int64_t batch, void *stream)
    {
        if (m && m->model.contactPoints().empty())
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "the model has no contact points (grbda_cuda_set_contact_points)");
        grbda_status st = vjpCheck(m, batch);
        if (st != GRBDA_OK || batch == 0)
            return st;
        if (!p_bar || !v_bar)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "null input pointer");
        DeviceScope scope(m->device);
        if (scope.error != cudaSuccess)
            return cudaFail(scope.error, "cudaSetDevice");
        const size_t n = 3 * m->model.contactPoints().size();
        double *packed = nullptr;
        if ((st = packRows(m, p_bar, n, v_bar, n, batch, (cudaStream_t)stream, packed)) != GRBDA_OK)
            return st;
        return launchAlgo(m, compiler::ALGO_CONTACT_KIN_VJP, false, q, yd, packed, q_bar, yd_bar, nullptr, batch, stream);
    }
    grbda_status grbda_cuda_contact_forward_dynamics_f64(const grbda_model *m, const double *q, const double *yd,
                                                         const double *tau, const uint8_t *active, double damping,
                                                         double *ydd, double *lambda, int64_t batch, void *stream)
    {
        return launchContact(m, compiler::ALGO_CONTACT_FD, q, yd, tau, active, 0.0, damping, ydd, lambda, batch, stream);
    }
    grbda_status grbda_cuda_contact_impulse_f64(const grbda_model *m, const double *q, const double *yd,
                                                const uint8_t *active, double restitution, double damping,
                                                double *yd_plus, double *impulse, int64_t batch, void *stream)
    {
        return launchContact(m, compiler::ALGO_CONTACT_IMPULSE, q, yd, nullptr, active, restitution, damping, yd_plus,
                             impulse, batch, stream);
    }
    grbda_status grbda_cuda_inverse_osim_f64(const grbda_model *m, const double *q, double *lambda_inv, int64_t batch,
                                             void *stream)
    {
        if (m && m->model.getNumEndEffectors() == 0)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "the model has no end-effectors (grbda_cuda_set_contact_points)");
        return launchAlgo(m, compiler::ALGO_OSIM, false, q, nullptr, nullptr, lambda_inv, nullptr, nullptr, batch, stream);
    }

    // ---- integration step / simulation step (SURVEY 8 f2) ---------------------------------------------------
    grbda_status grbda_cuda_integrate_f64(const grbda_model *m, const double *q, const double *yd, const double *ydd,
                                          double dt, double *q_out, double *yd_out, int32_t *flags, int64_t batch,
                                          void *stream)
    {
        if (!m || !q || !yd || !ydd || !q_out || !yd_out || batch < 0)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad arguments");
        if (m->device < 0 || !m->hasKernels())
            return fail(GRBDA_ERR_NO_DEVICE, "model was created without a CUDA device (host-only handle)");
        if (m->kernels && !m->kernels->integrate)
            return fail(GRBDA_ERR_NOT_COMPILED, "integration step was not compiled for this model");
        DeviceScope scope(m->device);
        if (scope.error != cudaSuccess)
            return cudaFail(scope.error, "cudaSetDevice");
        grbda_runtime::StepArgs a{q, yd, ydd, dt, batch, q_out, yd_out, flags, (cudaStream_t)stream};
        if (m->jit)
        {
            std::string err;
            if (!grbda_runtime::jitPrepareGenerate(*m->jit, m->model, m->hash, m->device, err))
                return fail(GRBDA_ERR_NOT_COMPILED, "integration step: " + err);
        }
        const cudaError_t e = m->jit ? grbda_runtime::jitLaunchIntegrate(m->jit->generate, a) : m->kernels->integrate(a);
        if (e != cudaSuccess)
            return cudaFail(e, "integrate launch");
        g_launches++;
        return GRBDA_OK;
    }

    grbda_status grbda_cuda_step_f64(const grbda_model *m, const double *q, const double *yd, const double *tau,
                                     const double *f_ext, double dt, double *q_out, double *yd_out, int32_t *flags,
                                     int64_t batch, void *stream)
    {
        if (!m || batch < 0)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad arguments");
        if (batch == 0)
            return GRBDA_OK;
        if (m->device < 0 || !m->hasKernels())
            return fail(GRBDA_ERR_NO_DEVICE, "model was created without a CUDA device (host-only handle)");
        const size_t bytes = (size_t)batch * m->model.getNumDegreesOfFreedom() * sizeof(double);
        double *ydd = (double *)m->scratchFor((cudaStream_t)stream, bytes, 2);
        if (!ydd)
            return fail(GRBDA_ERR_CUDA, "cannot allocate the acceleration buffer: " + m->scratch_error);
        grbda_status st = grbda_cuda_forward_dynamics_ext_f64(m, q, yd, tau, f_ext, ydd, batch, stream);
        if (st != GRBDA_OK)
            return st;
        return grbda_cuda_integrate_f64(m, q, yd, ydd, dt, q_out, yd_out, flags, batch, stream);
    }

    // ---- reverse mode of the integration step / simulation step -----------------------------------------------
    grbda_status grbda_cuda_integrate_vjp_f64(const grbda_model *m, const double *q, const double *yd, const double *ydd,
                                              double dt, const double *q_out_bar, const double *yd_out_bar,
                                              double *q_bar, double *yd_bar, double *ydd_bar, int32_t *flags,
                                              int64_t batch, void *stream)
    {
        grbda_status st = vjpCheck(m, batch);
        if (st != GRBDA_OK || batch == 0)
            return st;
        if (!q || !yd || !ydd || !q_out_bar || !yd_out_bar)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "null input pointer");
        if (!q_bar || !yd_bar || !ydd_bar)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "null output pointer");
        DeviceScope scope(m->device);
        if (scope.error != cudaSuccess)
            return cudaFail(scope.error, "cudaSetDevice");
        ensureExtJit(m);
        std::string err;
        if (!grbda_runtime::jitPrepareIntegrateVjp(*m->jit_ext, m->model, m->device, err))
            return fail(GRBDA_ERR_NOT_COMPILED, "reverse integration step: " + err);
        const grbda_runtime::StepVjpArgs a{q, yd, ydd, dt, q_out_bar, yd_out_bar, batch, q_bar, yd_bar, ydd_bar, flags,
                                           (cudaStream_t)stream};
        const cudaError_t e = grbda_runtime::jitLaunchIntegrateVjp(m->jit_ext->integrate_vjp, a);
        if (e != cudaSuccess)
            return cudaFail(e, "integrate vjp launch");
        g_launches++;
        return GRBDA_OK;
    }

    grbda_status grbda_cuda_step_vjp_f64(const grbda_model *m, const double *q, const double *yd, const double *tau,
                                         const double *f_ext, double dt, const double *q_out_bar, const double *yd_out_bar,
                                         double *q_bar, double *yd_bar, double *tau_bar, double *f_bar, int32_t *flags,
                                         int64_t batch, void *stream)
    {
        grbda_status st = vjpCheck(m, batch);
        if (st != GRBDA_OK || batch == 0)
            return st;
        if (!q || !yd || !tau || !q_out_bar || !yd_out_bar)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "null input pointer");
        if (!q_bar || !yd_bar || !tau_bar || (f_ext && !f_bar))
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "null output pointer");
        DeviceScope scope(m->device);
        if (scope.error != cudaSuccess)
            return cudaFail(scope.error, "cudaSetDevice");
        const cudaStream_t s = (cudaStream_t)stream;
        const int64_t nq = m->model.getNumPositions(), nv = m->model.getNumDegreesOfFreedom();
        double *ydd = (double *)m->scratchFor(s, (size_t)(batch * nv) * sizeof(double), 2);
        double *bars = (double *)m->scratchFor(s, (size_t)(batch * (nq + 2 * nv)) * sizeof(double), 5);
        if (!ydd || !bars)
            return fail(GRBDA_ERR_CUDA, "cannot allocate the step scratch buffers: " + m->scratch_error);
        double *q_bar_int = bars, *yd_bar_int = bars + batch * nq, *ydd_bar = yd_bar_int + batch * nv;
        if ((st = grbda_cuda_forward_dynamics_ext_f64(m, q, yd, tau, f_ext, ydd, batch, stream)) != GRBDA_OK ||
            (st = grbda_cuda_integrate_vjp_f64(m, q, yd, ydd, dt, q_out_bar, yd_out_bar, q_bar_int, yd_bar_int, ydd_bar,
                                               flags, batch, stream)) != GRBDA_OK ||
            (st = grbda_cuda_forward_dynamics_ext_vjp_f64(m, q, yd, tau, f_ext, ydd_bar, q_bar, yd_bar, tau_bar, f_bar,
                                                          batch, stream)) != GRBDA_OK)
            return st;
        return accumulate(q_bar, q_bar_int, batch * nq, yd_bar, yd_bar_int, batch * nv, s);
    }

    // ---- host placement for the host-buffer path ------------------------------------------------------------
    // One process per GPU pulls its states out of pinned host memory: that memory and the threads that feed the
    // copies should sit on the NUMA node the GPU's PCIe root hangs off, otherwise every byte crosses the socket
    // interconnect (measured: the 8-GPU end-to-end rate collapses when all ranks allocate on node 0).
    grbda_status grbda_cuda_bind_host_to_device(int device, int32_t *info4)
    {
        int32_t local[4] = {-1, 0, 0, 0}; // {numa node, cpus bound, memory policy set, cpus allowed before}
        int32_t *info = info4 ? info4 : local;
        std::memcpy(info, local, sizeof(local));
        char bus[64] = {0};
        cudaError_t e = cudaDeviceGetPCIBusId(bus, sizeof(bus), device);
        if (e != cudaSuccess)
            return cudaFail(e, "cudaDeviceGetPCIBusId");
        std::string id = bus;
        for (char &c : id)
            c = (char)std::tolower((unsigned char)c);
        int node = -1;
        {
            std::ifstream f("/sys/bus/pci/devices/" + id + "/numa_node");
            if (!(f >> node))
                node = -1;
        }
        info[0] = node;
        if (node < 0)
            return GRBDA_OK; // single-node machine or no information: nothing to bind
        // cpus of that node that this process may use
        cpu_set_t allowed, want;
        CPU_ZERO(&allowed);
        CPU_ZERO(&want);
        if (sched_getaffinity(0, sizeof(allowed), &allowed) != 0)
            return GRBDA_OK;
        info[3] = CPU_COUNT(&allowed);
        std::string list;
        {
            std::ifstream f("/sys/devices/system/node/node" + std::to_string(node) + "/cpulist");
            std::getline(f, list);
        }
        std::stringstream ss(list);
        std::string item;
        while (std::getline(ss, item, ','))
        {
            int a = 0, b = 0;
            if (std::sscanf(item.c_str(), "%d-%d", &a, &b) == 2)
                ;
            else if (std::sscanf(item.c_str(), "%d", &a) == 1)
                b = a;
            else
                continue;
            for (int c = a; c <= b && c < CPU_SETSIZE; c++)
                if (CPU_ISSET(c, &allowed))
                    CPU_SET(c, &want);
        }
        if (CPU_COUNT(&want) > 0 && sched_setaffinity(0, sizeof(want), &want) == 0)
            info[1] = CPU_COUNT(&want);
        // prefer the node for every later allocation of this thread (pinned buffers are first touched by the driver
        // in the allocating thread): MPOL_PREFERRED = 1
        unsigned long mask[16] = {0};
        if (node < (int)(sizeof(mask) * 8))
        {
            mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
            if (syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, mask, sizeof(mask) * 8) == 0)
                info[2] = 1;
        }
        return GRBDA_OK;
    }

    // ---- states, checks, measurement -----------------------------------------------------------------
    grbda_status grbda_cuda_generate_states(const grbda_model *m, uint64_t seed, int64_t first_index,
                                            int64_t count, double *q, double *yd, double *aux, int32_t *flags,
                                            void *stream)
    {
        if (!m || !q || !yd || !aux || count < 0)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad arguments");
        if (m->device < 0 || !m->hasKernels())
            return fail(GRBDA_ERR_NO_DEVICE, "model was created without a CUDA device (host-only handle)");
        if (m->kernels && !m->kernels->generate)
            return fail(GRBDA_ERR_NOT_COMPILED, "state generator was not compiled for this model");
        DeviceScope scope(m->device);
        if (scope.error != cudaSuccess)
            return cudaFail(scope.error, "cudaSetDevice");
        grbda_runtime::GenArgs a{seed, first_index, count, q, yd, aux, flags, (cudaStream_t)stream};
        if (m->jit)
        {
            std::string err;
            if (!grbda_runtime::jitPrepareGenerate(*m->jit, m->model, m->hash, m->device, err))
                return fail(GRBDA_ERR_NOT_COMPILED, "state generator: " + err);
        }
        cudaError_t e = m->jit ? grbda_runtime::jitLaunchGenerate(m->jit->generate, a) : m->kernels->generate(a);
        if (e != cudaSuccess)
            return cudaFail(e, "generate launch");
        g_launches++;
        return GRBDA_OK;
    }

    grbda_status grbda_cuda_constraint_violation_f64(const grbda_model *m, const double *q, double *max_abs_phi,
                                                     int64_t batch, void *stream)
    {
        if (!m || !q || !max_abs_phi)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad arguments");
        if (m->device < 0 || !m->hasKernels())
            return fail(GRBDA_ERR_NO_DEVICE, "model was created without a CUDA device (host-only handle)");
        DeviceScope scope(m->device);
        if (scope.error != cudaSuccess)
            return cudaFail(scope.error, "cudaSetDevice");
        cudaStream_t st = (cudaStream_t)stream;
        struct
        {
            int n_in[3], n_out[3];
        } ak;
        if (!entrySizes(m, compiler::ALGO_PHI, false, ak.n_in, ak.n_out))
        {
            // no implicit cluster: violation is zero by definition
            cudaError_t e = cudaMemsetAsync(max_abs_phi, 0, batch * 8, st);
            return e == cudaSuccess ? GRBDA_OK : cudaFail(e, "cudaMemsetAsync");
        }
        double *phi = nullptr, *Kd = nullptr;
        cudaError_t e = cudaMallocAsync(&phi, (size_t)batch * ak.n_out[0] * 8, st);
        if (e != cudaSuccess)
            return cudaFail(e, "cudaMallocAsync");
        e = cudaMallocAsync(&Kd, (size_t)batch * ak.n_out[1] * 8, st);
        if (e != cudaSuccess)
            return cudaFail(e, "cudaMallocAsync");
        grbda_status rs = launchAlgo(m, compiler::ALGO_PHI, false, q, nullptr, nullptr, phi, Kd, nullptr, batch, stream);
        if (rs == GRBDA_OK && batch > 0)
        {
            grbda_kernels::rowMaxAbsKernel<<<(unsigned)((batch + 127) / 128), 128, 0, st>>>(phi, ak.n_out[0], batch,
                                                                                           max_abs_phi);
            e = cudaGetLastError();
            if (e != cudaSuccess)
                rs = cudaFail(e, "rowMaxAbsKernel");
            g_launches++;
        }
        cudaFreeAsync(phi, st);
        cudaFreeAsync(Kd, st);
        return rs;
    }

    grbda_status grbda_cuda_checksum_f64(const double *x, int64_t n, double *out2, void *stream)
    {
        if (!x || !out2 || n < 0)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "bad arguments");
        cudaStream_t st = (cudaStream_t)stream;
        double *d = nullptr;
        cudaError_t e = cudaMallocAsync(&d, 16, st);
        if (e != cudaSuccess)
            return cudaFail(e, "cudaMallocAsync");
        cudaMemsetAsync(d, 0, 16, st);
        if (n > 0)
        {
            const int grid = (int)std::min<int64_t>((n + 255) / 256, 148 * 8);
            grbda_kernels::checksumKernel<<<grid, 256, 0, st>>>(x, n, d);
            g_launches++;
        }
        e = cudaMemcpyAsync(out2, d, 16, cudaMemcpyDeviceToHost, st);
        cudaFreeAsync(d, st);
        if (e == cudaSuccess)
            e = cudaStreamSynchronize(st);
        return e == cudaSuccess ? GRBDA_OK : cudaFail(e, "checksum");
    }

    grbda_status grbda_cuda_measure_fma_peak(int device, int fp32, double seconds, double *flops_per_s)
    {
        if (!flops_per_s)
            return fail(GRBDA_ERR_INVALID_ARGUMENT, "null output");
        cudaError_t e = cudaSetDevice(device);
        if (e != cudaSuccess)
            return cudaFail(e, "cudaSetDevice");
        cudaDeviceProp prop;
        cudaGetDeviceProperties(&prop, device);
        const int grid = prop.multiProcessorCount * 8, block = 256, iters = 4096;
        void *out = nullptr;
        cudaMalloc(&out, 64);
        cudaEvent_t t0, t1;
        cudaEventCreate(&t0);
        cudaEventCreate(&t1);
        double best = 0.0, elapsed = 0.0;
        for (int rep = 0; rep < 200 && (rep < 5 || elapsed < seconds); rep++)
        {
            cudaEventRecord(t0);
            if (fp32)
                grbda_kernels::fmaPeakKernel<float><<<grid, block>>>((float *)out, iters, 1.0000001f, 1e-7f);
            else
                grbda_kernels::fmaPeakKernel<double><<<grid, block>>>((double *)out, iters, 1.0000001, 1e-7);
            cudaEventRecord(t1);
            e = cudaEventSynchronize(t1);
            if (e != cudaSuccess)
                break;
            g_launches++;
            float ms = 0;
            cudaEventElapsedTime(&ms, t0, t1);
            elapsed += ms * 1e-3;
            const double flops = 2.0 * 64.0 * iters * (double)grid * block;
            if (rep >= 2)
                best = std::max(best, flops / (ms * 1e-3));
        }
        cudaEventDestroy(t0);
        cudaEventDestroy(t1);
        cudaFree(out);
        if (e != cudaSuccess)
            return cudaFail(e, "fma peak");
        *flops_per_s = best;
        return GRBDA_OK;
    }

    int64_t grbda_cuda_launch_count(void) { return g_launches.load(); }
}
