// ctcb_proj.cu -- translation unit of the tcgen05 projection kernel (ctcb_proj.cuh) and its launcher.
#define CTCB_PROJ_IMPL
#define CTCB_NO_PLAIN_KERNELS
#include "ctcb_proj.cuh"

namespace ctcb {

cudaError_t launch_proj_emit(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, const ProjArgs& a, int mode, dim3 grid,
                             size_t smem, cudaStream_t stream, bool programmatic) {
    // the opt-in shared-memory size is a per-device function attribute: raised when a launch needs more than any before
    static thread_local int done_dev = -1;
    static thread_local size_t done_bytes[16] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (done_dev != dev) { done_dev = dev; for (size_t& d : done_bytes) d = 0; }
    const int pair = a.ctas == 2 ? 1 : 0, bf = a.bf16 ? 1 : 0, which = mode * 4 + pair * 2 + bf;
    using Fn = void (*)(CUtensorMap, CUtensorMap, CUtensorMap, ProjArgs);
#define PROJ_MODE(M_) k_proj_emit<1, false, M_>, k_proj_emit<1, true, M_>, k_proj_emit<2, false, M_>, k_proj_emit<2, true, M_>
    static const Fn fns[16] = {PROJ_MODE(kProjLoss), PROJ_MODE(kProjLossDecode), PROJ_MODE(kProjDecode), PROJ_MODE(kProjGrad)};
#undef PROJ_MODE
    const Fn fn = fns[which];
    if (done_bytes[which] < smem) {
        const cudaError_t rc = cudaFuncSetAttribute(reinterpret_cast<const void*>(fn), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (rc != cudaSuccess) return rc;
        done_bytes[which] = smem;
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = dim3(kPThreads); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    int na = 0;
    if (pair) {
        attr[na].id = cudaLaunchAttributeClusterDimension;
        attr[na].val.clusterDim.x = 2; attr[na].val.clusterDim.y = 1; attr[na].val.clusterDim.z = 1;
        ++na;
    }
    if (programmatic) {
        attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[na].val.programmaticStreamSerializationAllowed = 1;
        ++na;
    }
    cfg.attrs = attr; cfg.numAttrs = na;
    const cudaError_t rc = cudaLaunchKernelEx(&cfg, fn, tmA, tmB, tmC, a);
    if (rc != cudaSuccess) return rc;
    return cudaGetLastError();
}

cudaError_t launch_proj_occ(const Problem& p, const Workspace& w, cudaStream_t stream) {
    const dim3 grid(p.B, (w.NB + kOccBlocksPerCta - 1) / kOccBlocksPerCta);
    k_proj_occ<<<grid, kOccThreads, 0, stream>>>(p, w);
    return cudaGetLastError();
}

}  // namespace ctcb
