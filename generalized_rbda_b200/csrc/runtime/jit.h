// Run-time model compilation: a model that was not compiled ahead of time (build.py MODELS) gets its
// kernels from the same model compiler + the same hand-written shells, built for sm_100a by NVRTC the
// first time an entry point is used and cached on disk (GRBDA_CACHE_DIR, default ~/.cache/grbda_cuda).
// Replaces nothing in the reference (it interprets any model at run time); it is what makes
// grbda_cuda_model_create / _from_urdf work for ARBITRARY ClusterTreeModels
// (reference: include/grbda/Dynamics/ClusterTreeModel.h:33-53, src/Dynamics/ClusterTreeParsing.cpp:5-43).
#pragma once
#include <cuda_runtime.h>
#include <memory>
#include <mutex>
#include <string>
#include "../compiler/compile.h"
#include "registry.h"

namespace grbda_runtime
{
    // launch shape the run-time compiler picks for one entry point (the ahead-of-time table of build.py
    // lists the same fields per model)
    struct JitShape
    {
        char kind = 'T'; // 'T' bulk-copy staged tiles, 'D' direct global I/O (rows do not fit into an SM)
        int block = 128, min_blocks = 2;
        int program = 0;
        bool park = false;
        bool slow_staged = true;
        size_t smem_fast = 0, smem_slow = 0, smem_unaligned = 0;
    };

    struct JitKernel
    {
        bool ready = false;
        std::string error; // non-empty: compilation failed before, do not retry
        JitShape shape;
        bool range_checked = false;
        int n_in[3] = {0, 0, 0}, n_out[3] = {0, 0, 0};
        int64_t counts[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        cudaLibrary_t library = nullptr;
        cudaKernel_t fast = nullptr;      // straight-line body, fast sin/cos
        cudaKernel_t slow = nullptr;      // flagged-tile pass (library sin/cos); also serves unaligned pointers
        bool from_cache = false;
        double compile_seconds = 0.0;
    };

    struct JitModel
    {
        std::mutex mutex;
        JitKernel algo[grbda::compiler::PROGRAM_COUNT][2]; // [entry point][0 f64, 1 f32] (slot 7 unused)
        JitKernel generate;
        JitKernel integrate_vjp; // reverse integration step (jitIntegrateVjpSource)
    };

    // Arguments of grbda_integrate_vjp_kernel (kernels/stategen.cuh)
    struct StepVjpArgs
    {
        const double *q, *yd, *ydd;
        double dt;
        const double *q_out_bar, *yd_out_bar;
        int64_t count;
        double *q_bar, *yd_bar, *ydd_bar;
        int32_t *flags;
        cudaStream_t stream;
    };

    // GRBDA_JIT: "0" never compile at run time, "force" ignore the ahead-of-time registry (tests), else: on a registry miss
    int jitMode(); // 0 off, 1 on miss, 2 force

    // Shape only (sizes and counts), no compilation; false + error if the entry point does not exist for this
    // model (phi without implicit clusters).
    bool jitDescribe(const grbda::ClusterTreeModel &model, int algo, bool f32, JitKernel &k, std::string &error);
    // Compile (or load from the cache) and load onto `device`. Thread-safe per JitModel.
    bool jitPrepare(JitModel &jm, const grbda::ClusterTreeModel &model, uint64_t model_hash, int device, int algo,
                    bool f32, std::string &error);
    bool jitPrepareGenerate(JitModel &jm, const grbda::ClusterTreeModel &model, uint64_t model_hash, int device,
                            std::string &error);
    bool jitPrepareIntegrateVjp(JitModel &jm, const grbda::ClusterTreeModel &model, int device, std::string &error);
    cudaError_t jitLaunch(const JitKernel &k, bool f32, const LaunchArgs &a);
    cudaError_t jitLaunchGenerate(const JitKernel &k, const GenArgs &a);
    cudaError_t jitLaunchIntegrate(const JitKernel &k, const StepArgs &a); // k = JitModel::generate (second kernel of that module)
    cudaError_t jitLaunchIntegrateVjp(const JitKernel &k, const StepVjpArgs &a); // k = JitModel::integrate_vjp
    void jitRelease(JitModel &jm);

    // The CUDA text handed to NVRTC for one entry point (tests compile it without a device).
    std::string jitSource(const grbda::ClusterTreeModel &model, int algo, bool f32, JitKernel &k,
                          std::vector<std::string> &name_expressions);
    std::string jitGenerateSource(const grbda::ClusterTreeModel &model, std::vector<std::string> &name_expressions);
    std::string jitIntegrateVjpSource(const grbda::ClusterTreeModel &model, std::vector<std::string> &name_expressions);
    // NVRTC only (no device needed): cubin + lowered names. `log` receives the compiler log on failure.
    bool jitCompile(const std::string &source, const std::vector<std::string> &name_expressions,
                    std::vector<char> &cubin, std::vector<std::string> &lowered, std::string &log);
} // namespace grbda_runtime
