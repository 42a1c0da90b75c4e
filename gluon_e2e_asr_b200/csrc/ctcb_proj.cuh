// ctcb_proj.cuh -- the output projection fused with the loss's emission stage (SURVEY.md section 8f, rank 1).
//
// Reference: /root/reference/scripts/swbd/model.py:394-398 (`tgt_proj = nn.Dense(units=V, flatten=False)`) and
// :424 (`return self.tgt_proj(net_out)`), whose output is the `pred` of CtcLoss (train_ctc_ce.py:363).  For the
// BPE-sized vocabulary (V = 2000) the logits are 8 KB per frame against 2 KB of encoder output: the tensor that
// dominates the step's HBM traffic is the one nobody needs -- the loss reads, per frame, the row maximum, the
// softmax normaliser and the L+1 columns of the utterance's own labels.
//
// k_proj_emit computes  logits[b, t, :] = hidden[b, t, :] . W^T + bias  on the 5th-generation tensor cores and
// reduces each 128-frame x 256-symbol accumulator tile to exactly those three things while it is still in tensor
// memory:
//   * one CTA per (utterance, 128-frame tile); the vocabulary is swept in tiles of 256 columns, the hidden units
//     in blocks of 32 fp32 values (= one 128-byte swizzle row);
//   * warp 0 (one lane): TMA producer -- `cp.async.bulk.tensor` of the A tile (3-D map over hidden (K, T, B): rows
//     beyond T are zero-filled by the hardware and never read the next utterance) and the B tile (2-D map over W
//     (K, V): rows beyond V zero-filled) into a 3-stage 128B-swizzled shared-memory ring, full/empty mbarriers;
//   * warp 1 (one lane): `tcgen05.mma.cta_group::1.kind::tf32`, M = 128, N = 256, K = 8 per instruction, fp32
//     accumulators in tensor memory, two accumulator stages (2 x 256 columns = the SM's whole TMEM) so that the
//     tensor cores work on vocabulary tile n+1 while the epilogue drains tile n; `tcgen05.commit` hands shared-memory
//     stages back to the producer and accumulator stages to the epilogue;
//   * warps 2..5: epilogue, ONE FRAME PER THREAD (TMEM lane = accumulator row): `tcgen05.ld.32x32b.x32` brings 32
//     columns of the thread's own row into registers; bias add, online row maximum / sum of exp2 (no shuffles: a
//     thread owns its row), optional store of the logits row chunk for the gradient kernel (training) -- or no
//     store at all (validation, train_ctc_ce.py:143: the logits never exist in HBM).  The store goes through a
//     128B-swizzled 32 x 32 staging tile per warp and leaves with `cp.async.bulk.tensor` (TMA store, 3-D map over the
//     logits: rows beyond T and columns beyond V are clipped by the hardware) -- a thread owns a ROW, so direct
//     stores would write 16 bytes per row and instruction (measured: +90 us at V = 2000);
//   * the utterance's label columns that fall into the tile are fetched again from TMEM with single-column loads
//     (the column index is uniform over the warp) and parked, raw, in their slot of the emission table E;
//   * after the sweep every thread writes its frame's {row max, log2 sum} to `fr` and turns its parked columns into
//     the softmax numerators relative to the final row maximum (fp64, frame-minor blocks of 8 frames) -- `fr` and E
//     are the two inputs of k_walk's unfused variant, bit-compatible with what k_emit writes from a logits tensor.
// The tf32 data path reads the caller's fp32 tensors as they are (the tensor cores ignore the low 13 mantissa
// bits): no conversion pass, no copy of hidden or W.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "ctcb_kernels.cuh"

namespace ctcb {

constexpr int kPM = 128;                 // frames per CTA tile = UMMA M (TMEM lanes)
constexpr int kPN = 256;                 // vocabulary columns per accumulator stage = UMMA N
constexpr int kPK = 32;                  // fp32 values per K block: 128 bytes, one SWIZZLE_128B row
__host__ __device__ constexpr int proj_stages(int ctas) { return ctas == 2 ? 4 : 3; }    // shared-memory ring depth
constexpr int kPEpiWarps = 8;             // two epilogue warps per TMEM lane quadrant: each takes half of a tile's columns
constexpr int kPThreads = 64 + 32 * kPEpiWarps;   // warp 0 TMA, warp 1 MMA + TMEM allocation, warps 2.. epilogue
constexpr uint32_t kPBytesA = kPM * kPK * 4;     // 16 KB
constexpr uint32_t kPBytesB = kPN * kPK * 4;     // 32 KB (a CTA pair: each CTA stages half of it)
__host__ __device__ constexpr uint32_t proj_stage_bytes(int ctas) { return kPBytesA + kPBytesB / ctas; }
constexpr uint32_t kPTmemCols = 512;             // two accumulator stages of kPN columns

struct ProjArgs {
    Problem p; Workspace w;
    const float* bias;       // (V,) or nullptr
    float* logits;           // where the projection's output is kept for the gradient kernel (Problem::logits), or nullptr
    int K, NT, KB;           // hidden units, vocabulary tiles, K blocks
    int vec4;                // bias allows 16-byte loads
    int store;               // 0: logits not stored; 1: TMA store through the staging tiles; 2: direct scalar stores
                             //   (kProjGrad: the gradient, 1 = TMA store, 2 = coalesced row stores from the staging tiles)
    int smem_stash;          // the label columns are parked in shared memory (store == 0 and they fit), else in E
    int ctas;                // 1: one CTA per tile; 2: CTA pairs (tcgen05 cta_group::2) over 256 frames
    int bf16;                // operands are bfloat16 (64 values per 128-byte K block, kind::f16) instead of fp32 (32, kind::tf32)
    int dbg;                 // measurement only (option proj_dbg): 1 = the epilogue skips its arithmetic (results are garbage)
    int* tok;                // DECODE: (B, T) one word per valid frame -- the symbol after the <unk> rule, bit 31 set when the
                             //   raw best symbol is `unk` -- collapsed into the hypothesis by k_greedy_collapse
    int unk;                 // DECODE: the <unk> index, or -1 for no <unk> rule
};

constexpr uint32_t kPStageTile = 32 * 32 * 4;    // one warp's 32 frames x 32 columns on their way to the logits tensor
// the region behind the ring: staging tiles of the logits store, or -- when the logits are not stored and the label
// row fits -- the parked label columns [Lmax+1][128] (otherwise they are parked in the emission table itself)
__host__ __device__ inline bool proj_smem_stash(int Lmax, bool store) { return !store && (size_t)(Lmax + 1) * kPM * sizeof(float) <= 80 * 1024; }
__host__ __device__ inline size_t proj_side_bytes(int Lmax, bool store) {
    if (store) return (size_t)kPEpiWarps * 2 * kPStageTile;
    return proj_smem_stash(Lmax, store) ? (size_t)(Lmax + 1) * kPM * sizeof(float) : 0;
}
// decode: + the upper column halves' top-2 lists, where the two halves of a row meet
__host__ __device__ inline size_t proj_smem_bytes(int Lmax, int Lp, bool store, int NT, int ctas, bool decode = false) {
    return 1024 + (size_t)proj_stages(ctas) * proj_stage_bytes(ctas) + proj_side_bytes(Lmax, store) +
           (size_t)Lp * sizeof(int) + 128 + 2 * kPM * sizeof(float2) + (size_t)(Lp + 4) * sizeof(int) + (size_t)(2 * NT + 4) * sizeof(int) +
           (decode ? kPM * sizeof(Top2) : 0);
}

// what k_proj_emit's epilogue computes (its MODE, see there)
enum : int { kProjLoss = 0, kProjLossDecode = 1, kProjDecode = 2, kProjGrad = 3 };

// The occupancy table O of the recomputing training path (ctcb_proj_forward with keep_for_backward and no logits buffer):
// gamma_t(j) = sum over the lattice states of column j (0 = blank, j = label j) of alpha_t(s) beta'_t(s) / P(l|x), fp32, in
// E's frame-minor (B, NB, W, kEC) index space.  It lives in E's region: the walkers are the last readers of E, and the
// occupancy kernel runs after them in stream order.  Written by k_proj_occ, read by k_proj_emit<..., kProjGrad>.
__host__ __device__ inline float* proj_occ_table(const Workspace& w) { return reinterpret_cast<float*>(w.E); }
// frame blocks per CTA of k_proj_occ (each CTA forms P(l|x) once for all of them)
constexpr int kOccBlocksPerCta = 16;
constexpr int kOccThreads = 256;
constexpr int kGradOcc = 8;               // kProjGrad: occupancies of a chunk's label columns in flight per round trip

// (a.ctas == 2: grid.x even, launched as clusters of two CTAs along x)
// host-side launcher, defined in ctcb_proj.cu (its own translation unit: the kernel below is compiled there only)
// mode: kProjLoss, kProjLossDecode or kProjDecode (what the epilogue computes, see k_proj_emit)
// programmatic: launched with programmatic stream serialization (it starts beside the kernel enqueued before it)
cudaError_t launch_proj_emit(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, const ProjArgs& a, int mode, dim3 grid,
                             size_t smem, cudaStream_t stream, bool programmatic);
// k_proj_occ over the batch (an ordinary launch: the walkers before it in the stream have completed)
cudaError_t launch_proj_occ(const Problem& p, const Workspace& w, cudaStream_t stream);

#ifdef CTCB_PROJ_IMPL
// ---- tcgen05 / TMA wrappers -------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// CTA pair: each CTA loads its own tiles, the transaction bytes are counted on the LEADER's mbarrier (`bar` is the
// barrier's address with the pair's rank bit cleared)
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_3d_pair(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
constexpr uint32_t kPairRankMask = 0xFEFFFFFFu;   // shared::cluster address of the same offset in the pair's even CTA
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPairRankMask) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
// shared -> global tile store (the staging tile was written with ordinary stores: the caller fences the proxy)
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* tm, uint32_t src, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                 ::"l"(tm), "r"(src), "r"(c0), "r"(c1), "r"(c2) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(tm) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t slot_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_smem), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// CTA pair: the same warp of BOTH CTAs allocates (and frees), with the same shared-memory slot offset
__device__ __forceinline__ void tmem_alloc_pair(uint32_t slot_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_smem), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// D[tmem] (+)= A[smem] . B[smem]^T, tf32 inputs, fp32 accumulation; issued by ONE thread for the CTA
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// CTA pair: M = 256 (128 rows from each CTA's A tile), B = the two CTAs' halves, D in each CTA's own tensor memory;
// issued by one thread of the LEADER CTA for both SMs
__device__ __forceinline__ void umma_tf32_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// ... and the completion arrives on the mbarrier at the same offset in BOTH CTAs
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"((uint16_t)3) : "memory");
}
// the same two with bfloat16 operands (kind::f16: 16 values = 32 bytes of K per instruction, twice the rate)
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrives on the mbarrier when every tcgen05.mma issued so far by this thread has completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ uint32_t tmem_ld1(uint32_t taddr) {
    uint32_t v;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(v) : "r"(taddr) : "memory");
    return v;
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// shared-memory matrix descriptor of a K-major tile whose rows are 128 bytes (one SWIZZLE_128B row per row,
// 8-row groups 1024 bytes apart) -- the layout TMA writes with CU_TENSOR_MAP_SWIZZLE_128B.  Bits: [0,14) start
// address >> 4, [16,30) leading byte offset >> 4 (unused for swizzled K-major), [32,46) stride byte offset >> 4,
// [46,48) descriptor version 1 (sm_100), [61,64) layout type 2 = SWIZZLE_128B.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(1024u >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// instruction descriptor: D fp32 (bit 4), A and B tf32 (format 2 at bits 7 and 10), both K-major, N >> 3 at
// bit 17, M >> 4 at bit 24
constexpr uint32_t kPIdesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(kPN >> 3) << 17) | ((uint32_t)(kPM >> 4) << 24);
constexpr uint32_t kPIdescPair = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(kPN >> 3) << 17) | ((uint32_t)((2 * kPM) >> 4) << 24);
// bfloat16 operands: format 1 at bits 7 and 10
constexpr uint32_t kPIdescBf = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kPN >> 3) << 17) | ((uint32_t)(kPM >> 4) << 24);
constexpr uint32_t kPIdescBfPair = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kPN >> 3) << 17) | ((uint32_t)((2 * kPM) >> 4) << 24);

__device__ __forceinline__ void bar_sync_epilogue() { asm volatile("bar.sync 1, %0;" ::"n"(32 * kPEpiWarps) : "memory"); }

// What the epilogue makes of the tiles (MODE):
//   kProjLoss        the loss's inputs: {row max, normaliser} in `fr`, the label columns in E, the tile flags;
//   kProjLossDecode  the same, and each frame's row is also reduced to its best and second best symbol (k_greedy_decode's
//                    order: greater value, ties to the lower index) for the frame's word of ProjArgs::tok -- the greedy
//                    decode of the logits that are never stored;
//   kProjDecode      the frame's word only (ctcb_proj_greedy_decode: no labels): label parsing, the label columns, the
//                    normaliser, `fr`, E and the tile flags are compiled out, the word is the kProjLossDecode one;
//   kProjGrad        d loss / d logits of the recomputing training path (ctcb_proj_backward): the product is formed again,
//                    tile by tile, and each element becomes  head[b] * (softmax - occupancy)  with the forward's `fr` row and
//                    the occupancy table O (proj_occ_table) -- the logits are never written or read.  The label columns of a
//                    half tile are sorted by symbol, so those of one 32-column chunk are a contiguous run; their
//                    occupancies are fetched while the chunk's softmax is formed and subtracted, in fp32, in the staging
//                    tile before it leaves (TMA tile store into p.grad, or coalesced row stores when p.grad's rows do
//                    not allow a tensor map).  Tiles of padded frames, infeasible utterances and a workspace that no
//                    matching forward filled skip the product: zeros (NaN for the last) are written instead.
// A compile-time switch: a run-time branch in this kernel was measured at +17 us (DESIGN.md section 5)
template <int CTAS, bool BF16, int MODE>
__global__ void __launch_bounds__(kPThreads, 1)
k_proj_emit(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmC,
            ProjArgs a) {
    constexpr bool LOSS = MODE == kProjLoss || MODE == kProjLossDecode, DECODE = MODE == kProjLossDecode || MODE == kProjDecode;
    constexpr bool GRAD = MODE == kProjGrad, LABELS = LOSS || GRAD;
    extern __shared__ unsigned char proj_raw[];
    __shared__ int s_L;
    const Problem& p = a.p;
    const Workspace& w = a.w;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // grid (CTAS, B, tiles / CTAS): the utterances' first tiles (pairs) are scheduled before anybody's second -- a recursion
    // kernel that runs beside this one (its programmatic dependent) can start on the first frames of every utterance
    const int b = blockIdx.y, mt = (int)blockIdx.z * CTAS + (int)blockIdx.x, m0 = mt * kPM;

    // the metadata kernel behind this one in the stream is its programmatic dependent: it needs nothing from here and
    // runs in this kernel's shadow (its small CTAs fit beside a resident projection CTA)
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // operator parameter layer, frame count: lengths truncated and clamped (as k_emit does)
    int Tb = p.T;
    if (p.data_len) {
        long long t64 = load_as_int(p.data_len, p.data_len_dtype, b);
        t64 = t64 < 0 ? 0 : (t64 > p.T ? p.T : t64);
        Tb = (int)t64;
    }
    if constexpr (GRAD) {
        // rows without a product: the tile (pair) lies beyond Tb, the utterance is infeasible (G = 0), or no matching forward
        // filled the workspace (G = NaN, never a wait).  The words read are the utterance's, so both CTAs of a pair agree
        const bool filled = __ldcg(w.gprog + 4 * b + 2) == w.stamp && __ldcg(w.gprog + 4 * b + 3) == w.stamp;
        const bool zero = !filled || (CTAS == 2 ? (int)blockIdx.z * 2 * kPM : m0) >= Tb || (__ldcg(w.flags + b) & UTT_INFEASIBLE);
        if (zero) {
            if (warp < 2) return;
            // the epilogue warps: a quadrant's two warps take alternate rows of its 32, all V columns, coalesced
            const float fill = filled ? 0.0f : __int_as_float(0x7fc00000);
            for (int rr = (warp - 2) >> 2; rr < 32; rr += 2) {
                const int t = m0 + (warp & 3) * 32 + rr;
                if (t >= p.T) break;
                float* grow = p.grad + (long long)b * p.gst_b + (long long)t * p.gst_t;
                for (int v = lane; v < p.V; v += 32) grow[v] = fill;
            }
            return;
        }
    }
    // a tile of padded frames: nothing of it is ever read (a pair leaves together: its second CTA stages half of B)
    if ((CTAS == 2 ? (int)blockIdx.z * 2 * kPM : m0) >= Tb) return;
    constexpr int kPStages = proj_stages(CTAS);
    constexpr uint32_t kBytesB = kPBytesB / CTAS;
    const uint32_t rank = CTAS == 2 ? cluster_ctarank() : 0u;

    const uint32_t raw = smem_u32(proj_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;          // SWIZZLE_128B tiles want 1024-byte alignment
    unsigned char* gbase = proj_raw + (base - raw);
    const uint32_t sA = base, sB = base + kPStages * kPBytesA;
    const uint32_t sC = base + kPStages * (kPBytesA + kBytesB);           // [epilogue warp][2] staging tiles of the logits store
    float* stash = reinterpret_cast<float*>(gbase + (size_t)kPStages * (kPBytesA + kBytesB));    // [Lmax+1][128], a.smem_stash only
    int* labs = reinterpret_cast<int*>(gbase + (size_t)kPStages * (kPBytesA + kBytesB) + proj_side_bytes(p.Lmax, a.store != 0));
    uint64_t* bars = reinterpret_cast<uint64_t*>(labs + w.Lp);
    uint64_t* full = bars;
    uint64_t* empty = bars + kPStages;
    uint64_t* tfull = bars + 2 * kPStages;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
    float2* part = reinterpret_cast<float2*>(bars + 16);                 // [2][128] {row max, sum} of each column half
    int* order = reinterpret_cast<int*>(part + 2 * kPM);                  // lattice columns 0..L sorted by half tile of their symbol
    int* hstart = order + w.Lp + 4;                                       // [2 NT + 1] where each half tile's columns start in `order`

    if (tid == 0) {
        for (int s = 0; s < kPStages; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(tfull + s, 1); mbar_init(tempty + s, CTAS * 32 * kPEpiWarps); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        s_L = p.Lmax;
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        if (a.store == 1) tma_prefetch_desc(&tmC);
    }
    if (warp == 1) { if (CTAS == 2) tmem_alloc_pair(smem_u32(tmem_slot), kPTmemCols); else tmem_alloc(smem_u32(tmem_slot), kPTmemCols); }
    tc_fence_before();
    if (CTAS == 2) cluster_sync_all(); else __syncthreads();      // the pair's barriers exist before anything arrives on them
    tc_fence_after();
    const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(tmem_slot);

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            int st = 0; uint32_t ph = 0;
            constexpr int kelems = BF16 ? 2 * kPK : kPK;        // values per 128-byte K block
            for (int n = 0; n < a.NT; ++n)
                for (int kb = 0; kb < a.KB; ++kb) {
                    mbar_wait(empty + st, ph ^ 1u);
                    if (CTAS == 2) {
                        // both CTAs' bytes are counted on the leader's barrier; this CTA stages its own 128 frames and its
                        // half of the vocabulary tile
                        if (rank == 0) mbar_expect_tx(full + st, 2 * (kPBytesA + kBytesB));
                        const uint32_t lbar = smem_u32(full + st) & kPairRankMask;
                        tma_load_3d_pair(sA + st * kPBytesA, &tmA, lbar, kb * kelems, m0, b);
                        tma_load_2d_pair(sB + st * kBytesB, &tmB, lbar, kb * kelems, n * kPN + (int)rank * (kPN / 2));
                    } else {
                        mbar_expect_tx(full + st, kPBytesA + kBytesB);
                        tma_load_3d(sA + st * kPBytesA, &tmA, smem_u32(full + st), kb * kelems, m0, b);
                        tma_load_2d(sB + st * kBytesB, &tmB, smem_u32(full + st), kb * kelems, n * kPN);
                    }
                    if (++st == kPStages) { st = 0; ph ^= 1u; }
                }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (a pair: its leader CTA, for both SMs) =====
        if (lane == 0 && rank == 0) {
            int st = 0; uint32_t ph = 0;
            for (int n = 0; n < a.NT; ++n) {
                const int as = n & 1;
                mbar_wait(tempty + as, (((uint32_t)n >> 1) & 1u) ^ 1u);       // the epilogue has drained this accumulator stage
                tc_fence_after();
                const uint32_t dcol = tmem + (uint32_t)as * kPN;
                for (int kb = 0; kb < a.KB; ++kb) {
                    mbar_wait(full + st, ph);
                    tc_fence_after();
                    const uint32_t a0 = sA + st * kPBytesA, b0 = sB + st * kBytesB;
#pragma unroll
                    for (int k = 0; k < kPK / 8; ++k) {                        // 32 bytes of K per instruction: 8 tf32 or 16 bf16 values
                        const uint64_t da = umma_desc_sw128(a0 + k * 32), db = umma_desc_sw128(b0 + k * 32);
                        const uint32_t acc = (uint32_t)((kb | k) != 0);
                        if (BF16) { if (CTAS == 2) umma_bf16_pair(dcol, da, db, kPIdescBfPair, acc); else umma_bf16(dcol, da, db, kPIdescBf, acc); }
                        else { if (CTAS == 2) umma_tf32_pair(dcol, da, db, kPIdescPair, acc); else umma_tf32(dcol, da, db, kPIdesc, acc); }
                    }
                    // the stage is free (in both CTAs) once these MMAs have read it
                    if (CTAS == 2) umma_commit_pair(smem_u32(empty + st)); else umma_commit(smem_u32(empty + st));
                    if (++st == kPStages) { st = 0; ph ^= 1u; }
                }
                // the accumulator tile is complete (in both CTAs' tensor memory)
                if (CTAS == 2) umma_commit_pair(smem_u32(tfull + as)); else umma_commit(smem_u32(tfull + as));
            }
        }
    } else {
        // ===== epilogue: one frame per thread pair (each thread takes half of a tile's columns) =====
        constexpr int NE = 32 * kPEpiWarps;
        constexpr int HC = kPN / 2;                   // columns per thread and tile
        const int etid = tid - 64;
        const int q = warp & 3;                       // TMEM lane quadrant this warp may read
        const int hsel = (warp - 2) >> 2;             // which half of the tile's columns
        const int r = q * 32 + lane;                  // accumulator row = frame within the tile
        const int t = m0 + r;
        if constexpr (LABELS) {
            // labels (the rest of the parameter layer; bad labels are clamped here and reported by the metadata CTA)
            int L;
            if (p.label_len) {
                long long l64 = load_as_int(p.label_len, p.label_len_dtype, b);
                l64 = l64 < 0 ? 0 : (l64 > p.Lmax ? p.Lmax : l64);
                L = (int)l64;
            } else {
                for (int j = etid; j < p.Lmax; j += NE)
                    if (load_as_int(p.labels, p.label_dtype, b * p.lst_b + j * p.lst_l) == p.label_pad) atomicMin(&s_L, j);
                bar_sync_epilogue();
                L = s_L;
            }
            for (int j = etid; j < L; j += NE) {
                const long long v = load_as_int(p.labels, p.label_dtype, b * p.lst_b + j * p.lst_l);
                labs[j] = (int)(v < 0 ? 0 : (v >= p.V ? p.V - 1 : v));
            }
            bar_sync_epilogue();
            // the lattice's columns (0 = blank, j = label j) bucketed by the half tile (128 symbols) their symbol lies in, the
            // buckets of the lower column halves first (key = half * NT + tile): an epilogue warp visits exactly its own
            // columns of a tile, and all the columns a thread parks are one contiguous range of `order`
            for (int h = etid; h <= 2 * a.NT; h += NE) {
                int c = 0;
                for (int j = 0; j <= L; ++j) { const int hb = (j == 0 ? p.blank : labs[j - 1]) >> 7; c += ((hb & 1) * a.NT + (hb >> 1)) < h; }
                hstart[h] = c;
            }
            for (int j = etid; j <= L; j += NE) {
                const int sj = j == 0 ? p.blank : labs[j - 1], hb = sj >> 7;
                const int key = (hb & 1) * a.NT + (hb >> 1);
                int pos = 0;
                for (int k = 0; k <= L; ++k) {
                    const int sk = k == 0 ? p.blank : labs[k - 1], hk = sk >> 7;
                    const int kk = (hk & 1) * a.NT + (hk >> 1);
                    // GRAD: within a bucket by symbol, then position (a chunk's columns are one run of `order`)
                    if constexpr (GRAD) pos += (kk < key) | ((kk == key) & ((sk < sj) | ((sk == sj) & (k < j))));
                    else pos += (kk < key) | ((kk == key) & (k < j));
                }
                order[pos] = j;
            }
            bar_sync_epilogue();
        }
        // GRAD: this frame's softmax row ({row max, log2 normaliser} of the forward), head, and its slots of O
        float2 gfr = make_float2(0.0f, 0.0f);
        float ghead = 1.0f;
        const float* ocol = nullptr;
        if constexpr (GRAD) {
            if (t < Tb) gfr = __ldcg(w.fr + (size_t)b * p.T + t);
            ghead = p.head ? __ldg(p.head + b) : 1.0f;
            ocol = proj_occ_table(w) + ((size_t)b * w.NB + (t < Tb ? (t >> 3) : 0)) * w.W * kEC + (t & 7);
        }
        int gk = 0;                                   // GRAD: the next of this half tile's label columns in `order`

        float* lrow = (LOSS && a.store == 2 && t < p.T) ? a.logits + (long long)b * p.st_b + (long long)t * p.st_t : nullptr;
        // this frame's slots of the emission table (block of 8 frames, frame-minor): parked raw, finished below
        const int blk = t >> 3;
        const bool eblock = blk < w.NB && blk * kG < Tb;
        const bool valid = t < Tb;
        double* ecol = w.E + ((size_t)b * w.NB + (eblock ? blk : 0)) * w.W * kEC + (t & 7);
        const uint32_t sbuf = sC + (uint32_t)(warp - 2) * 2 * kPStageTile;
        int nstored = 0;
        float mx = -INFINITY, sum = 0.0f;
        Top2 tp{-INFINITY, 0x7fffffff, -INFINITY, 0x7fffffff};   // DECODE: the best two of this thread's columns
        for (int n = 0; n < a.NT; ++n) {
            const int as = n & 1;
            mbar_wait(tfull + as, ((uint32_t)n >> 1) & 1u);
            tc_fence_after();
            const uint32_t trow = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * kPN + hsel * HC);
            const int cbase = n * kPN + hsel * HC;
            uint32_t v[2][32];
            if (a.dbg & 1) { tc_fence_before(); if (CTAS == 2) mbar_arrive_leader(tempty + as); else mbar_arrive(tempty + as); continue; }
            if (cbase < p.V) tmem_ld32(trow, v[0]);
            const int gend = GRAD ? hstart[hsel * a.NT + n + 1] : 0;
            if constexpr (GRAD) gk = hstart[hsel * a.NT + n];
            // one chunk of 32 columns; FULLC: every column lies below V (no bounds checks: all but the vocabulary's last chunks)
            auto chunk = [&](auto full_tag, const int c, const int col0) {
                constexpr bool FULLC = decltype(full_tag)::value;
                tmem_ld_wait();
                // the next chunk's accumulators travel while this one is reduced
                if (c + 1 < HC / 32 && col0 + 32 < p.V) tmem_ld32(trow + (c + 1) * 32, v[(c + 1) & 1]);
                float x[32];
                if (a.vec4) {
#pragma unroll
                    for (int i = 0; i < 32; i += 4) {
                        const bool in = FULLC || col0 + i < p.V;                // V % 4 == 0: whole groups
                        const float4 bb = (in && a.bias) ? __ldg(reinterpret_cast<const float4*>(a.bias + col0 + i)) : make_float4(0.f, 0.f, 0.f, 0.f);
                        x[i] = in ? __uint_as_float(v[c & 1][i]) + bb.x : -INFINITY;
                        x[i + 1] = in ? __uint_as_float(v[c & 1][i + 1]) + bb.y : -INFINITY;
                        x[i + 2] = in ? __uint_as_float(v[c & 1][i + 2]) + bb.z : -INFINITY;
                        x[i + 3] = in ? __uint_as_float(v[c & 1][i + 3]) + bb.w : -INFINITY;
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        const bool in = FULLC || col0 + i < p.V;
                        x[i] = in ? __uint_as_float(v[c & 1][i]) + (a.bias ? __ldg(a.bias + col0 + i) : 0.0f) : -INFINITY;
                    }
                }
                if constexpr (GRAD) {
                    // the chunk's label columns are order[gk, gk1): their occupancies travel while the softmax is formed
                    auto sym = [&](int j) { return j == 0 ? p.blank : labs[j - 1]; };
                    int gk1 = gk;
                    while (gk1 < gend && sym(order[gk1]) < col0 + 32) ++gk1;
                    float ov[kGradOcc];
#pragma unroll
                    for (int i = 0; i < kGradOcc; ++i) ov[i] = (valid && gk + i < gk1) ? __ldcg(ocol + (size_t)order[gk + i] * kEC) : 0.0f;
                    // head * softmax, k_grad's arithmetic (padded rows: 0; columns >= V: ex2(-inf) = 0)
#pragma unroll
                    for (int i = 0; i < 32; ++i) x[i] = valid ? ghead * fast_ex2(fmaf(x[i] - gfr.x, kLog2e, -gfr.y)) : 0.0f;
                    const uint32_t tile = sbuf + (uint32_t)(nstored & 1) * kPStageTile;
                    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");   // the store that read this tile two chunks ago
                    __syncwarp();
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};"
                                     ::"r"(tile + (uint32_t)lane * 128u + (uint32_t)((i ^ (lane & 7)) << 4)),
                                       "f"(x[4 * i]), "f"(x[4 * i + 1]), "f"(x[4 * i + 2]), "f"(x[4 * i + 3]) : "memory");
                    // minus head * occupancy in the thread's own row (a repeated symbol: once per lattice column)
                    float* trowp = reinterpret_cast<float*>(gbase + (tile - base)) + lane * 32;
                    for (int k0 = gk; k0 < gk1; k0 += kGradOcc) {
                        if (k0 != gk) {
#pragma unroll
                            for (int i = 0; i < kGradOcc; ++i) ov[i] = (valid && k0 + i < gk1) ? __ldcg(ocol + (size_t)order[k0 + i] * kEC) : 0.0f;
                        }
#pragma unroll
                        for (int i = 0; i < kGradOcc; ++i)
                            if (k0 + i < gk1) {
                                const int ci = sym(order[k0 + i]) - col0;
                                float* e = trowp + (((ci >> 2) ^ (lane & 7)) << 2) + (ci & 3);
                                *e = fmaf(-ghead, ov[i], *e);
                            }
                    }
                    gk = gk1;
                    if (a.store == 1) {
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        __syncwarp();
                        if (lane == 0) tma_store_3d(&tmC, tile, col0, m0 + q * 32, b);
                    } else {
                        // rows whose strides allow no tensor map: the warp writes the tile row by row, 128 bytes at a time
                        __syncwarp();
                        const float* tf = reinterpret_cast<const float*>(gbase + (tile - base));
                        for (int rr = 0; rr < 32; ++rr) {
                            const int t2 = m0 + q * 32 + rr;
                            if (t2 >= p.T) break;
                            if (FULLC || col0 + lane < p.V)
                                p.grad[(long long)b * p.gst_b + (long long)t2 * p.gst_t + col0 + lane] =
                                    tf[rr * 32 + ((((lane >> 2) ^ (rr & 7))) << 2) + (lane & 3)];
                        }
                        __syncwarp();
                    }
                    ++nstored;
                    return;
                }
                if (LOSS && a.store == 1 && !(a.dbg & 2)) {
                    // 32 frames x 32 columns through a swizzled staging tile: row = lane, 16-byte chunk i at (i ^ row % 8)
                    const uint32_t tile = sbuf + (uint32_t)(nstored & 1) * kPStageTile;
                    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");   // the store that read this tile two chunks ago
                    __syncwarp();
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};"
                                     ::"r"(tile + (uint32_t)lane * 128u + (uint32_t)((i ^ (lane & 7)) << 4)),
                                       "f"(x[4 * i]), "f"(x[4 * i + 1]), "f"(x[4 * i + 2]), "f"(x[4 * i + 3]) : "memory");
                    if (!(a.dbg & 8)) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) tma_store_3d(&tmC, tile, col0, m0 + q * 32, b);
                    ++nstored;
                } else if (lrow) {
#pragma unroll
                    for (int i = 0; i < 32; ++i)
                        if (FULLC || col0 + i < p.V) lrow[col0 + i] = x[i];
                }
                float cm[4] = {x[0], x[1], x[2], x[3]};
#pragma unroll
                for (int i = 4; i < 32; i += 4) {
                    cm[0] = fmaxf(cm[0], x[i]); cm[1] = fmaxf(cm[1], x[i + 1]);
                    cm[2] = fmaxf(cm[2], x[i + 2]); cm[3] = fmaxf(cm[3], x[i + 3]);
                }
                const float cmx = fmaxf(fmaxf(cm[0], cm[1]), fmaxf(cm[2], cm[3]));
                // the normaliser (kProjDecode: mx and sum are never read, and the compiler drops this)
                if (cmx > mx) { sum *= fast_ex2((mx - cmx) * kLog2e); mx = cmx; }     // first chunk: mx = -inf -> sum (0) * 0
                const float ms = mx * kLog2e;
                float sp[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
                for (int i = 0; i < 32; i += 4) {
                    sp[0] += fast_ex2(fmaf(x[i], kLog2e, -ms));
                    sp[1] += fast_ex2(fmaf(x[i + 1], kLog2e, -ms));
                    sp[2] += fast_ex2(fmaf(x[i + 2], kLog2e, -ms));
                    sp[3] += fast_ex2(fmaf(x[i + 3], kLog2e, -ms));
                }
                sum += (sp[0] + sp[1]) + (sp[2] + sp[3]);
                if constexpr (DECODE) {
                    // a thread visits its columns in increasing order: a chunk whose maximum only ties the second best
                    // holds higher indices and cannot displace it (one compare per 32 columns in the common case).
                    // Columns >= V are never pushed
                    if (cmx > tp.v2 || tp.i2 == 0x7fffffff) {
#pragma unroll
                        for (int i = 0; i < 32; ++i)
                            if (FULLC || col0 + i < p.V) top2_push(tp, x[i], col0 + i);
                    }
                }
            };
#pragma unroll
            for (int c = 0; c < HC / 32; ++c) {
                const int col0 = cbase + c * 32;
                if (col0 + 32 <= p.V) chunk(std::true_type{}, c, col0);          // warp-uniform
                else if (col0 < p.V) chunk(std::false_type{}, c, col0);
            }
            // the utterance's own columns in this half tile (blank, l_1..l_L): column index uniform over the warp
            if constexpr (LOSS) {
                for (int k = hstart[hsel * a.NT + n]; k < hstart[hsel * a.NT + n + 1]; ++k) {
                    const int j = order[k];
                    const int vj = j == 0 ? p.blank : labs[j - 1];
                    const uint32_t raw1 = tmem_ld1(trow + (uint32_t)(vj & (HC - 1)));
                    tmem_ld_wait();
                    const float xv = __uint_as_float(raw1) + (a.bias ? __ldg(a.bias + vj) : 0.0f);
                    if (a.smem_stash) stash[j * kPM + r] = xv;
                    else if (eblock && !(a.dbg & 4)) ecol[(size_t)j * kEC] = valid ? (double)xv : 0.0;
                }
            }
            tc_fence_before();
            if (CTAS == 2) mbar_arrive_leader(tempty + as); else mbar_arrive(tempty + as);
        }
        if constexpr (GRAD) { if (a.store == 1 && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }   // tiles read before exit
        // ---- the two column halves of a row meet: row max and normaliser ----
        if constexpr (LOSS) part[hsel * kPM + r] = make_float2(mx, sum);
        Top2* htop = reinterpret_cast<Top2*>(hstart + 2 * a.NT + 4);      // DECODE: [128] the upper halves' top-2 lists
        if constexpr (DECODE) { if (hsel == 1) htop[r] = tp; }
        bar_sync_epilogue();
        if constexpr (LOSS) {
            const float2 o = part[(hsel ^ 1) * kPM + r];
            const float m2 = fmaxf(mx, o.x);           // a half without columns holds {-inf, 0}: ex2(-inf) = 0
            sum = sum * fast_ex2((mx - m2) * kLog2e) + o.y * fast_ex2((o.x - m2) * kLog2e);
            mx = m2;
        }
        if constexpr (DECODE) {
            // the frame's word: the best symbol, or the second best when the best is `unk` (k_greedy_decode's rule and
            // fallback); bit 31 keeps the raw best for the repeat test of the next frame, whatever V is
            if (hsel == 0 && valid) {
                const Top2 o = htop[r];
                top2_push(tp, o.v1, o.i1);
                top2_push(tp, o.v2, o.i2);
                const bool is_unk = a.unk >= 0 && tp.i1 == a.unk;
                const int sym = (is_unk && tp.i2 != 0x7fffffff) ? tp.i2 : tp.i1;
                a.tok[(size_t)b * p.T + t] = sym | (is_unk ? (int)0x80000000 : 0);
            }
        }
        if constexpr (LOSS) {
            // ---- the frame's outputs: {row max, log2 normaliser}; the parked columns (each thread finishes the ones it
            // parked itself) become softmax numerators relative to the final row maximum ----
            if (hsel == 0 && valid) w.fr[(size_t)b * p.T + t] = make_float2(mx, log2f(sum));
            if (a.smem_stash) {
                if (eblock) {
                    bool floored = false;
                    for (int k = hstart[hsel * a.NT]; k < hstart[(hsel + 1) * a.NT]; ++k) {
                        const int j = order[k];
                        const float l2 = (stash[j * kPM + r] - mx) * kLog2e;
                        floored |= valid && l2 < kMinLog2;
                        ecol[(size_t)j * kEC] = valid ? (double)fast_ex2(fmaxf(l2, kMinLog2)) : 0.0;
                    }
                    if (floored && p.status) atomicOr(p.status + b, UTT_WIDE_LOGITS);
                }
            } else if (eblock && valid && !(a.dbg & 4)) {
                bool floored = false;
                const int k1 = hstart[(hsel + 1) * a.NT];
                for (int k0 = hstart[hsel * a.NT]; k0 < k1; k0 += 8) {          // eight independent round trips to L2 at a time
                    double raw[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        if (k0 + i < k1) raw[i] = ecol[(size_t)order[k0 + i] * kEC];
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        if (k0 + i < k1) {
                            const float l2 = ((float)raw[i] - mx) * kLog2e;
                            floored |= l2 < kMinLog2;
                            ecol[(size_t)order[k0 + i] * kEC] = (double)fast_ex2(fmaxf(l2, kMinLog2));
                        }
                }
                if (floored && p.status) atomicOr(p.status + b, UTT_WIDE_LOGITS);
            }
            if (a.store == 1 && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // staging tiles are read before the CTA exits
            // this tile's rows of `fr` and E are written: tell a recursion kernel that runs beside this one
            __threadfence();
            bar_sync_epilogue();
            if (etid == 0) st_release_gpu(w.tflag + (size_t)b * w.ntile + mt, 1);
        }
    }
    tc_fence_before();
    if (CTAS == 2) cluster_sync_all(); else __syncthreads();      // a pair: nobody leaves while its peer may still signal it
    if (warp == 1) { if (CTAS == 2) tmem_dealloc_pair(tmem, kPTmemCols); else tmem_dealloc(tmem, kPTmemCols); }
}

// k_proj_occ: the occupancy table O (proj_occ_table) from the walkers' α/β' history, the last kernel of the recomputing
// training forward.  grid (B, ceil(NB / kOccBlocksPerCta)), kOccThreads threads; it runs after the walkers in stream order.
// k_grad2's normalisation, with one prologue per CTA instead of one per frame block: warp 0 forms P(l|x) from the
// utterance's frame 0 (exact integer exponents, fp64 sum) as {exponent EP, 1 / mantissa}; a state's occupancy is then
// its stored alpha high word with the block's exponent shift (both walkers' offsets minus EP) added as an integer, one DMUL
// with beta's high word, times 1 / mantissa.  A warp takes whole frame blocks: lane g holds state pair g -- the blank state
// 2g, summed over the warp into column 0, and the label state 2g+1, column g+1 -- forms the pair's shift once per block and
// then covers the block's kG frames with all their history loads in flight.  Padded frames, columns beyond the utterance's
// labels and infeasible utterances get zeros.  The CTA of the first blocks stamps gprog word 3 (zeroed by every forward's
// metadata kernel) for ctcb_proj_backward.
__global__ void __launch_bounds__(kOccThreads) k_proj_occ(Problem p, Workspace w) {
    constexpr unsigned FULL = 0xffffffffu;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    __shared__ int s_EP;
    __shared__ float s_rP;
    float* O = proj_occ_table(w);
    const int Tb = __ldcg(w.Tb + b), Lb = __ldcg(w.Lb + b);
    const bool infeasible = (__ldcg(w.flags + b) & UTT_INFEASIBLE) != 0;
    const int NQ = infeasible ? 0 : (Tb + kG - 1) / kG;
    const int pairs = 32 * w.P * w.NW;
    const int blk0 = (int)blockIdx.y * kOccBlocksPerCta, blk1 = min(blk0 + kOccBlocksPerCta, w.NB);
    if (warp == 0 && blk0 < NQ) {
        // ---- P(l|x) = sum_s alpha_0(s) beta'_0(s), k_grad2's prologue over any number of state pairs ----
        const int2* hA0 = w.hA + (size_t)b * w.NB * kG * pairs;
        const int2* hB0 = w.hB + (size_t)b * w.NB * kG * pairs;
        const int2* oA = w.oA + (size_t)b * w.NB * pairs;
        const int2* oB = w.oB + (size_t)b * w.NB * pairs;
        auto term = [&](int g, int& exb, float& mb, int& exl, float& ml) {
            const int ib = Lb - g, il = max(Lb - 1 - g, 0);
            const int2 av = __ldcg(hA0 + g), oa = __ldcg(oA + g);
            const int hb = __ldcg(&hB0[ib].x), hl = __ldcg(&hB0[il].y);
            const int ob = __ldcg(&oB[ib].x), ol = __ldcg(&oB[il].y);
            const bool vb = av.x != 0 && hb != 0, vl = g < Lb && av.y != 0 && hl != 0;
            exb = vb ? (av.x >> 20) + (hb >> 20) - 2046 + oa.x + ob : INT_MIN / 2;
            exl = vl ? (av.y >> 20) + (hl >> 20) - 2046 + oa.y + ol : INT_MIN / 2;
            mb = vb ? hw_mant(av.x) * hw_mant(hb) : 0.0f;
            ml = vl ? hw_mant(av.y) * hw_mant(hl) : 0.0f;
        };
        int emax = INT_MIN / 2;
        for (int g = lane; g <= Lb; g += 32) {
            int eb, el; float mb, ml;
            term(g, eb, mb, el, ml);
            emax = max(emax, max(eb, el));
        }
        emax = __reduce_max_sync(FULL, emax);
        double s = 0.0;
        for (int g = lane; g <= Lb; g += 32) {
            int eb, el; float mb, ml;
            term(g, eb, mb, el, ml);
            s += (double)mb * pow2c(max(eb - emax, -2000));
            s += (double)ml * pow2c(max(el - emax, -2000));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
            s += __hiloint2double(__shfl_xor_sync(FULL, __double2hiint(s), o), __shfl_xor_sync(FULL, __double2loint(s), o));
        if (lane == 0) { s_EP = emax + dexp(s); s_rP = (float)(1.0 / dmant(s)); }
    }
    __syncthreads();
    const int EP = s_EP;
    const float rP = s_rP;
#pragma unroll 1
    for (int blk = blk0 + warp; blk < blk1; blk += kOccThreads / 32) {
        float* ob = O + ((size_t)b * w.NB + blk) * w.W * kEC;
        if (blk >= NQ) {
            for (int j = lane; j < w.W; j += 32)
#pragma unroll
                for (int f = 0; f < kG; ++f) ob[(size_t)j * kEC + f] = 0.0f;
            continue;
        }
        const size_t blkoff = (size_t)b * w.NB + blk;
        const int2* hA0 = w.hA + blkoff * kG * pairs;
        const int2* hB0 = w.hB + blkoff * kG * pairs;
        const int2* oA = w.oA + blkoff * pairs;
        const int2* oB = w.oB + blkoff * pairs;
        const int t_first = blk * kG;
        float zb[kG];
#pragma unroll
        for (int f = 0; f < kG; ++f) zb[f] = 0.0f;
        for (int g = lane; g < w.W; g += 32) {
            float zl[kG];
#pragma unroll
            for (int f = 0; f < kG; ++f) zl[f] = 0.0f;
            if (g <= Lb) {
                const int ib = Lb - g, il = max(Lb - 1 - g, 0);
                const int2 oa = __ldcg(oA + g);
                const int db = min(max(oa.x + __ldcg(&oB[ib].x) - EP, -2047), 2047);
                const int dl = min(max(oa.y + __ldcg(&oB[il].y) - EP, -2047), 2047);
                const int dsb = db * (1 << 20), dsl = g < Lb ? dl * (1 << 20) : INT_MIN;
                int2 av[kG]; int hb[kG], hl[kG];
#pragma unroll
                for (int f = 0; f < kG; ++f) {
                    const bool live = t_first + f < Tb;
                    av[f] = live ? __ldcg(hA0 + (size_t)f * pairs + g) : make_int2(0, 0);
                    hb[f] = live ? __ldcg(&hB0[(size_t)f * pairs + ib].x) : 0;
                    hl[f] = live ? __ldcg(&hB0[(size_t)f * pairs + il].y) : 0;
                }
#pragma unroll
                for (int f = 0; f < kG; ++f) {
                    // k_grad2's occupancy: an exact zero stays zero, a value that leaves the normal range is flushed
                    int tb = av[f].x != 0 ? (int)((unsigned)av[f].x + (unsigned)dsb) : 0;
                    int tl = av[f].y != 0 ? (int)((unsigned)av[f].y + (unsigned)dsl) : 0;
                    tb = tb < (1 << 20) ? 0 : tb; tl = tl < (1 << 20) ? 0 : tl;
                    zb[f] += (float)(__hiloint2double(tb, 0) * __hiloint2double(tb ? hb[f] : 0, 0));
                    zl[f] = (float)(__hiloint2double(tl, 0) * __hiloint2double(tl ? hl[f] : 0, 0)) * rP;
                }
            }
            if (g + 1 < w.W) {
#pragma unroll
                for (int f = 0; f < kG; ++f) ob[(size_t)(g + 1) * kEC + f] = zl[f];
            }
        }
#pragma unroll
        for (int f = 0; f < kG; ++f) zb[f] = warp_sum(zb[f]);
        if (lane == 0) {
#pragma unroll
            for (int f = 0; f < kG; ++f) ob[f] = zb[f] * rP;
        }
    }
    if (blockIdx.y == 0 && tid == 0) {
        __threadfence();
        st_release_gpu(w.gprog + 4 * b + 3, w.stamp);
    }
}

#endif  // CTCB_PROJ_IMPL

}  // namespace ctcb
