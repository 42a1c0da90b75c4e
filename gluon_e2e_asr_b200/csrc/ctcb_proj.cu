// ctcb_proj.cu -- translation unit of the tcgen05 projection kernel (ctcb_proj.cuh) and its launcher.
#define CTCB_PROJ_IMPL
#define CTCB_NO_PLAIN_KERNELS
#include "ctcb_proj.cuh"

namespace ctcb {

cudaError_t launch_proj_emit(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, const ProjArgs& a, int mode, dim3 grid,
                             size_t smem, cudaStream_t stream, bool programmatic) {
    const int pair = a.ctas == 2 ? 1 : 0, bf = a.bf16 ? 1 : 0, which = mode * 4 + pair * 2 + bf;
    using Fn = void (*)(CUtensorMap, CUtensorMap, CUtensorMap, ProjArgs);
#define PROJ_MODE(M_) k_proj_emit<1, false, M_>, k_proj_emit<1, true, M_>, k_proj_emit<2, false, M_>, k_proj_emit<2, true, M_>
    static const Fn fns[16] = {PROJ_MODE(kProjLoss), PROJ_MODE(kProjLossDecode), PROJ_MODE(kProjDecode), PROJ_MODE(kProjGrad)};
#undef PROJ_MODE
    const Fn fn = fns[which];
    if (cudaError_t rc = ensure_dynamic_smem(reinterpret_cast<const void*>(fn), smem)) return rc;
    if (cudaError_t rc = launch_ex(fn, grid, dim3(kPThreads), smem, stream, programmatic, pair ? 2 : 1, tmA, tmB, tmC, a)) return rc;
    return cudaGetLastError();
}

cudaError_t launch_proj_occ(const Problem& p, const Workspace& w, cudaStream_t stream) {
    const dim3 grid(p.B, (w.NB + kOccBlocksPerCta - 1) / kOccBlocksPerCta);
    k_proj_occ<<<grid, kOccThreads, 0, stream>>>(p, w);
    return cudaGetLastError();
}

}  // namespace ctcb
