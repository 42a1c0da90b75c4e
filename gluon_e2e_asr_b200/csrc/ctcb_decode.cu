// ctcb_decode.cu -- translation unit of the decoding variants of k_walk and k_emit (ctcb_forward_decode_typed): the loss
// evaluation that also leaves each valid frame's greedy-decode word for k_greedy_collapse.  Kept apart from ctcb.cu so that
// the two units compile side by side and the existing instantiations stay where they were.
#define CTCB_NO_PLAIN_KERNELS
#include "ctcb_kernels.cuh"

namespace ctcb {

WalkKernel walk_decode_kernel(int P, int NW, bool bf16) {
#define DECODE_WALK(P_, NW_) \
    if (P == P_ && NW == NW_) return bf16 ? k_walk<P_, NW_, false, true, ctcb::bf16, true> : k_walk<P_, NW_, false, true, float, true>;
    CTCB_WALK_CONFIGS(DECODE_WALK)
#undef DECODE_WALK
    return nullptr;
}

EmitKernel emit_decode_kernel(int vec, int nq, bool bf16) {
    if (nq < 0) return bf16 ? k_emit<4, -1, ctcb::bf16, true> : k_emit<4, -1, float, true>;
#define DECODE_EMIT_NQ(V_) \
    switch (nq) { \
        case 1: return bf16 ? k_emit<V_, 1, ctcb::bf16, true> : k_emit<V_, 1, float, true>; \
        case 2: return bf16 ? k_emit<V_, 2, ctcb::bf16, true> : k_emit<V_, 2, float, true>; \
        case 4: return bf16 ? k_emit<V_, 4, ctcb::bf16, true> : k_emit<V_, 4, float, true>; \
        case 8: return bf16 ? k_emit<V_, 8, ctcb::bf16, true> : k_emit<V_, 8, float, true>; \
        case 16: return bf16 ? k_emit<V_, 16, ctcb::bf16, true> : k_emit<V_, 16, float, true>; \
        default: return bf16 ? k_emit<V_, 0, ctcb::bf16, true> : k_emit<V_, 0, float, true>; \
    }
    switch (vec) {
        case 4: DECODE_EMIT_NQ(4)
        case 2: DECODE_EMIT_NQ(2)
        default: DECODE_EMIT_NQ(1)
    }
#undef DECODE_EMIT_NQ
}

}  // namespace ctcb
