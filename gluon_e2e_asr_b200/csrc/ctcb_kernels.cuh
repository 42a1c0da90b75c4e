// ctcb_kernels.cuh -- sm_100a device code of the CTC training-loss path.
//
// Path restated (SURVEY.md section 8a): softmax over V (row a4), blank-extended lattice
// (a5), alpha recursion (a6), beta recursion + per-label accumulation + gradient (a7),
// head-gradient scaling (a8) of `mx.nd.contrib.ctc_loss` as called at
// /root/reference/scripts/swbd/loss.py:134-139.  Not a port: the reference operator works
// in fp32 log space; these kernels work in the LINEAR domain on B200's full-rate FP64 pipe
// (64 DFMA/clk/SM, 8.5-clk latency, measured: scripts/ubench/dp.cu) with one integer
// exponent offset per lattice state that only changes when a state drifts by more than
// 2^128 -- no exp/log and no exponent arithmetic inside the T-sequential chain
// (DESIGN.md section 4).
//
// Kernels (one batch = three launches, all on the caller's stream):
//   k_emit<VEC>          per frame: max / log2-sum-exp of the logits row; per block of 8
//                        frames the emission table E[b][n][col][8] (fp64 softmax numerators,
//                        frame-minor, one contiguous TMA-streamable block): the whole row when
//                        V is small ("dense"), the gathered columns blank, l_1..l_L otherwise; plus the
//                        per-utterance metadata (lengths, int labels, repeats, feasibility,
//                        same-label chains for the gradient scatter).
//   k_walk<P,NW,HIST>    grid (B, 2): the alpha walker and the (reversed) beta walker of one
//                        utterance run concurrently on different SMs; E is staged through a
//                        shared-memory ring with cp.async.bulk (TMA) + mbarriers by a producer
//                        warp; P (blank,label) state pairs per lane, one 64-bit warp shuffle
//                        per step, no CTA barrier (skewed wavefront across warps).
//   k_grad<VEC,CH>       per frame: posterior state occupancy normalised per frame
//                        (gamma = alpha*beta'/Z_t), scatter to label columns, fused
//                        grad = head * (softmax - occupancy) written once, coalesced.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace ctcb {

constexpr int kG = 8;                  // walker steps per group (= frames per emission block)
constexpr int kEC = 10;                // doubles per emission column: 8 frames + 16 bytes of padding, so that
                                       // 128-bit shared loads of different columns spread over all banks
constexpr int kD = 100;                // largest exponent step between neighbouring states
constexpr int kDrift = 200;            // a state renormalises when it drifts past 2^+-kDrift
constexpr int kZeroE = -(1 << 28);     // "natural exponent" of an exactly-zero state
constexpr float kLog2e = 1.4426950408889634f;
constexpr double kLn2 = 0.6931471805599453094;
constexpr float kMinLog2 = -100.0f;    // clamp of one frame's log2-probability (7.9e-31)
constexpr int kMaxStages = 16;         // emission ring depth (blocks of kG frames), at most

enum : int { UTT_INFEASIBLE = 1, UTT_BAD_LABEL = 2, UTT_LEN_CLAMPED = 4, UTT_WIDE_LOGITS = 8 };
constexpr long long kSpinLimit = 4000000000LL;   // clocks (~2 s) a gradient CTA waits for the recursion kernel before giving up
enum : int { DT_I32 = 0, DT_I64 = 1, DT_F32 = 2, DT_F64 = 3 };

struct Problem {          // device view of ctcb_problem_t
    int T, B, V, Lmax, blank, label_pad;
    const float* logits; long long st_t, st_b;   // fp32, or bf16 in the kernels instantiated with LT = bf16
    const long long* row_off;        // optional: element offset of utterance b's frame 0 (packed, ragged logits); replaces b*st_b
    float* grad; long long gst_t, gst_b;         // the logits' element type
    const void* labels; int label_dtype; long long lst_b, lst_l;
    const void* data_len; int data_len_dtype;
    const void* label_len; int label_len_dtype;
    const float* head;
    float* loss; double* loss_sum; int* status;
};

// loss evaluation with walkers that meet in the middle (WalkArgs::meet): what a walker hands over at the meeting frame --
// per state pair the mantissas in [1,2) (0 for an exact zero) and the full exponents of its blank / label state
struct MeetSlot { double vb, vl; int ob, ol; };

struct Workspace {        // carved out of the caller's workspace by the host (ctcb.cu)
    int* Tb; int* Lb; int* flags;     // (B,)
    int* lab;                         // (B, Lp) int32 labels
    int* rank;                        // (B, Lp) rank of each label position in the order (label value, position)
    int2* dl;                         // (B, Lp+1) distinct labels in increasing order: {value, start
                                      //   of its run in rank order}; entry nd is the sentinel {-1, L}
    int* nd;                          // (B,) number of distinct labels
    float2* fr;                       // (B, T) {row max, log2 sum exp2((x-max)*log2e)}
    double* E;                        // (B, NB, W, kEC) emissions exp(x - rowmax) of frame block n = t / 8, frame-minor:
                                      //   dense -> column v; else column 0 blank, column j label j
    int2* hA;                         // (B, NB, 8, NW*PW) alpha_t {blank, label} of each state pair, relative to oA:
                                      //   the HIGH WORD of the walker's fp64 value (11-bit exponent, 20-bit mantissa)
    int2* hB;                         // same for beta'_t in the reversed walker's pair coordinates, relative to oB
    int2* oA;                         // (B, NB, NW*PW) exponent offsets {blank, label} valid for frame block n
    int2* oB;
    int2* runv;                       // (B, 64) small vocabularies (fused path): the run [start, end) of every symbol's label
                                      //   positions in rank order (empty for symbols the utterance does not use)
    int2* pinfo;                      // (B,) {exponent of P(l|x), bits of the float 1 / mantissa}: written by the gradient
                                      //   kernel's middle frame block (k_grad2), read by the utterance's other blocks
    int* gprog;                       // (B, 4) {frame blocks whose history is complete: alpha walker, beta walker;
                                      //   metadata ready (Tb, Lb, flags, rank, dl, nd); pinfo ready}: published with
                                      //   release/gpu scope, polled by the gradient CTAs
    MeetSlot* meet;                   // (B, 2, NW*PW) meeting-frame states of the alpha / beta walker (loss evaluation, WalkArgs::meet)
    double* meetlz;                   // (B, 2) each side's sum of log2(softmax denominator) over its frames
    int* meetcnt;                     // (B,) walker warps that have handed over (zeroed by the host before the launch)
    int* tflag;                       // (B, ntile) fused projection (ctcb_proj.cuh): 1 once the 128-frame tile's rows of `fr` and E are
                                      //   written -- polled by the recursion kernel when it runs beside the projection
    int ntile;
    int Lp, W, NB, dense, P, NW;      // PW = 32*P pairs per walker warp
    int poll_ns;                      // back-off of the gradient CTAs' polls of the walkers' progress words (<= 0: the kernels' defaults)
    int stamp;                        // nonzero hash of the call's shape and layout choices: the value of the
                                      //   "metadata ready" progress word, checked by the gradient CTAs (a workspace
                                      //   that no matching forward call filled is an error, not a hang)
    int fused;                        // emissions made by the walkers' producer warps (no k_emit, no E)
};

__device__ __forceinline__ long long load_as_int(const void* p, int dtype, long long i) {
    switch (dtype) {
        case DT_I32: return static_cast<const int*>(p)[i];
        case DT_I64: return static_cast<const long long*>(p)[i];
        case DT_F32: return static_cast<long long>(static_cast<const float*>(p)[i]);
        default:     return static_cast<long long>(static_cast<const double*>(p)[i]);
    }
}

// frame 0 of utterance b: strided (any T/B strides), or packed -- utterance b's valid frames stored back to back
template <typename LT = float>
__device__ __forceinline__ const LT* utt_logits(const Problem& p, int b) {
    return reinterpret_cast<const LT*>(p.logits) + (p.row_off ? __ldg(p.row_off + b) : b * p.st_b);
}

__device__ __forceinline__ float fast_ex2(float x) {
    float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- greedy decode (k_greedy_decode and the decoding variants of k_emit / k_walk) ----
// a frame's best two {value, index}: ties go to the lowest index, NaN never wins (better() is a total order on the
// non-NaN pairs, so the order in which a kernel visits the columns does not change the result)
struct Top2 { float v1; int i1; float v2; int i2; };
__device__ __forceinline__ bool better(float va, int ia, float vb, int ib) { return va > vb || (va == vb && ia < ib); }
__device__ __forceinline__ void top2_push(Top2& t, float v, int i) {
    if (better(v, i, t.v1, t.i1)) { t.v2 = t.v1; t.i2 = t.i1; t.v1 = v; t.i1 = i; }
    else if (better(v, i, t.v2, t.i2)) { t.v2 = v; t.i2 = i; }
}
// top2_push as selects: the decoding variants insert inside long unrolled bodies, where top2_push's branches would
// cost reconvergence regions and registers (the result is the same)
__device__ __forceinline__ void top2_insert(Top2& t, float v, int i) {
    const bool b1 = better(v, i, t.v1, t.i1), b2 = better(v, i, t.v2, t.i2);
    t.v2 = b1 ? t.v1 : (b2 ? v : t.v2); t.i2 = b1 ? t.i1 : (b2 ? i : t.i2);
    t.v1 = b1 ? v : t.v1;               t.i1 = b1 ? i : t.i1;
}
constexpr Top2 kTop2Empty{-INFINITY, 0x7fffffff, -INFINITY, 0x7fffffff};
// merges the lists of the lanes `o` apart.  two = false: the best symbol alone (no <unk> rule), half the shuffles
__device__ __forceinline__ void top2_merge_xor(Top2& tp, int o) {
    const float ov1 = __shfl_xor_sync(0xffffffffu, tp.v1, o), ov2 = __shfl_xor_sync(0xffffffffu, tp.v2, o);
    const int oi1 = __shfl_xor_sync(0xffffffffu, tp.i1, o), oi2 = __shfl_xor_sync(0xffffffffu, tp.i2, o);
    top2_push(tp, ov1, oi1);
    top2_push(tp, ov2, oi2);
}
__device__ __forceinline__ void top2_merge_xor(Top2& tp, int o, bool two) {
    const float ov1 = __shfl_xor_sync(0xffffffffu, tp.v1, o);
    const int oi1 = __shfl_xor_sync(0xffffffffu, tp.i1, o);
    if (two) {
        const float ov2 = __shfl_xor_sync(0xffffffffu, tp.v2, o);
        const int oi2 = __shfl_xor_sync(0xffffffffu, tp.i2, o);
        top2_insert(tp, ov1, oi1);
        top2_insert(tp, ov2, oi2);
    } else {
        const bool b = better(ov1, oi1, tp.v1, tp.i1);
        tp.v1 = b ? ov1 : tp.v1; tp.i1 = b ? oi1 : tp.i1;
    }
}
__device__ __forceinline__ void top2_warp_merge(Top2& tp, bool two) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) top2_merge_xor(tp, o, two);
}
// the word a decoding kernel leaves per valid frame for k_greedy_collapse: the symbol after the <unk> rule (the second
// best when the best is `unk`), bit 31 set when the raw best symbol is `unk` (k_proj_emit's DECODE epilogue writes the same)
__device__ __forceinline__ int decode_word(const Top2& tp, int unk) {
    const bool is_unk = unk >= 0 && tp.i1 == unk;
    const int sym = (is_unk && tp.i2 != 0x7fffffff) ? tp.i2 : tp.i1;
    return sym | (is_unk ? (int)0x80000000 : 0);
}
// where the decoding variants of k_emit / k_walk leave their words: tok (B, T), one word per valid frame; unk < 0: no rule
struct DecodeOut { int* tok; int unk; };

// ---- fp64 exponent-field helpers ------------------------------------------------------
__device__ __forceinline__ int dexp11(double v) { return (__double2hiint(v) >> 20) & 0x7ff; }   // biased
__device__ __forceinline__ int dexp(double v) { return dexp11(v) - 1023; }
__device__ __forceinline__ double dmant(double v) {            // v with its exponent replaced by 0: [1,2)
    return __hiloint2double((__double2hiint(v) & 0x000fffff) | 0x3ff00000, __double2loint(v));
}
// 2^d, exactly 0 for d <= -1023, 2^1023 for d >= 1023
__device__ __forceinline__ double pow2c(int d) {
    d = min(max(d, -1023), 1023);
    return __hiloint2double((d + 1023) << 20, 0);
}
__device__ __forceinline__ double shfl_up_f64(double v) {
    return __hiloint2double(__shfl_up_sync(0xffffffffu, __double2hiint(v), 1),
                            __shfl_up_sync(0xffffffffu, __double2loint(v), 1));
}
// float m * 2^d, exactly 0 below 2^-64 (m is a positive normal float, d <= a few)
__device__ __forceinline__ float xscale0(float m, int d) {
    return d < -64 ? 0.0f : __int_as_float(__float_as_int(m) + d * (1 << 23));
}

// ---------------------------------------------------------------------------------------
// k_emit<VEC>: grid (ceil(NB/4), B), block 128, dynamic smem Lp ints; one warp per block of
// kG = 8 frames.
//
// Rows a3/a4/a5 of SURVEY 8a in one launch: every CTA derives its utterance's lengths and
// int labels itself; per frame {row max, log2 sum} (kept for the gradient's softmax); per
// frame block the emission table in the frame-minor layout the walkers read with 128-bit
// shared-memory loads: E[b][n][col][j] = exp(x_{8n+j}(v_col) - max_v x_{8n+j}(v)), i.e. the
// softmax numerator -- the per-frame normaliser is common to all lattice states, cancels in
// the posteriors and re-enters the loss as sum_t log2(sum).  one extra CTA per utterance
// publishes the per-utterance metadata.
// ---------------------------------------------------------------------------------------
template <int VEC> struct VecT;
template <> struct VecT<1> { using type = float; };
template <> struct VecT<2> { using type = float2; };
template <> struct VecT<4> { using type = float4; };

template <int VEC>
__device__ __forceinline__ void vec_get(const typename VecT<VEC>::type& v, float (&o)[VEC]);
template <> __device__ __forceinline__ void vec_get<1>(const float& v, float (&o)[1]) { o[0] = v; }
template <> __device__ __forceinline__ void vec_get<2>(const float2& v, float (&o)[2]) { o[0] = v.x; o[1] = v.y; }
template <> __device__ __forceinline__ void vec_get<4>(const float4& v, float (&o)[4]) { o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w; }

template <int VEC> __device__ __forceinline__ typename VecT<VEC>::type vec_fill(float v);
template <> __device__ __forceinline__ float vec_fill<1>(float v) { return v; }
template <> __device__ __forceinline__ float2 vec_fill<2>(float v) { return make_float2(v, v); }
template <> __device__ __forceinline__ float4 vec_fill<4>(float v) { return make_float4(v, v, v, v); }

// ---- logits element type (the LT template argument of the kernels that read logits or write the gradient) ----
// float, or bf16: a bf16 logit is widened to fp32 exactly where it is loaded, everything after that is the fp32 path's
// arithmetic, and a gradient element is that fp32 value rounded ONCE to bf16 (round to nearest even) where it is stored.
// Problem::logits / Problem::grad then point at bf16 elements; strides and row offsets stay in elements.
using bf16 = __nv_bfloat16;
__device__ __forceinline__ float bf_lo(unsigned u) { return __uint_as_float(u << 16); }          // element 0 of a bf16 pair
__device__ __forceinline__ float bf_hi(unsigned u) { return __uint_as_float(u & 0xffff0000u); }  // element 1
__device__ __forceinline__ unsigned bf_rn(float x) { return (unsigned)__bfloat16_as_ushort(__float2bfloat16_rn(x)); }
__device__ __forceinline__ unsigned bf_pair(float a, float b) { return bf_rn(a) | (bf_rn(b) << 16); }

// VEC consecutive elements of type LT as one load / store: get widens to fp32, pack rounds fp32 values
template <typename LT, int VEC> struct LV {
    using type = typename VecT<VEC>::type;
    static __device__ __forceinline__ void get(const type& v, float (&o)[VEC]) { vec_get<VEC>(v, o); }
    static __device__ __forceinline__ type fill(float v) { return vec_fill<VEC>(v); }
    static __device__ __forceinline__ type pack(const float (&y)[VEC]) { type o; memcpy(&o, y, sizeof(o)); return o; }
};
template <> struct LV<bf16, 1> {
    using type = unsigned short;
    static __device__ __forceinline__ void get(const type& v, float (&o)[1]) { o[0] = bf_lo(v); }
    static __device__ __forceinline__ type fill(float v) { return (type)bf_rn(v); }
    static __device__ __forceinline__ type pack(const float (&y)[1]) { return (type)bf_rn(y[0]); }
};
template <> struct LV<bf16, 2> {
    using type = unsigned int;
    static __device__ __forceinline__ void get(const type& v, float (&o)[2]) { o[0] = bf_lo(v); o[1] = bf_hi(v); }
    static __device__ __forceinline__ type fill(float v) { return bf_pair(v, v); }
    static __device__ __forceinline__ type pack(const float (&y)[2]) { return bf_pair(y[0], y[1]); }
};
template <> struct LV<bf16, 4> {
    using type = uint2;
    static __device__ __forceinline__ void get(const type& v, float (&o)[4]) { o[0] = bf_lo(v.x); o[1] = bf_hi(v.x); o[2] = bf_lo(v.y); o[3] = bf_hi(v.y); }
    static __device__ __forceinline__ type fill(float v) { return make_uint2(bf_pair(v, v), bf_pair(v, v)); }
    static __device__ __forceinline__ type pack(const float (&y)[4]) { return make_uint2(bf_pair(y[0], y[1]), bf_pair(y[2], y[3])); }
};
// one element: read-only load widened to fp32 / store rounded from fp32
__device__ __forceinline__ float ldx(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ldx(const bf16* p) { return bf_lo(__ldg(reinterpret_cast<const unsigned short*>(p))); }
__device__ __forceinline__ void stx(float* p, float v) { *p = v; }
__device__ __forceinline__ float ldsx(const float* p) { return *p; }             // shared memory
__device__ __forceinline__ float ldsx(const bf16* p) { return bf_lo(*reinterpret_cast<const unsigned short*>(p)); }
__device__ __forceinline__ void stx(bf16* p, float v) { *reinterpret_cast<unsigned short*>(p) = (unsigned short)bf_rn(v); }
// gradient row (b, t) in the element type of the call
template <typename LT>
__device__ __forceinline__ LT* grad_row(const Problem& p, int b, int t) {
    return reinterpret_cast<LT*>(p.grad) + b * p.gst_b + (long long)t * p.gst_t;
}

// frames [0, n) of one utterance (frame t at logits + base + t * st_t), a warp per frame -- warp w of nw takes frames w,
// w + nw, ...: the frame's best two symbols, handed to emit(t, top2) in lane 0
template <typename LT, typename Emit>
__device__ __forceinline__ void greedy_frames(const LT* logits, long long base, long long st_t, int n, int V, int warp, int nw, int lane,
                                              Emit&& emit) {
    for (int t = warp; t < n; t += nw) {
        const LT* row = logits + base + t * st_t;
        Top2 tp = kTop2Empty;
        for (int v = lane; v < V; v += 32) top2_push(tp, ldx(row + v), v);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) top2_merge_xor(tp, o);
        if (lane == 0) emit(t, tp);
    }
}

__device__ __forceinline__ void st_release_gpu(int* p, int v);
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count);
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes);
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity);
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar);

// NQ = VEC-wide loads per lane that cover one logits row (power of two, <= 16): the rows of
// F = 16/NQ frames (at most 8) are held in registers, so every global load of those frames is
// in flight before the first reduction.  NQ = 0: rows too wide for registers, two passes.
// NQ = -1 (wide vocabularies, 16-byte aligned rows): the frame block's kG rows are fetched into shared
// memory by 1-D bulk copies (TMA) before the parameter layer runs -- 8 rows in flight per CTA, several
// CTAs per SM -- and row maximum, normaliser and the gathered emission columns all read shared memory:
// every logit crosses HBM exactly once.
__host__ __device__ constexpr int emit_blocks_per_cta(int nq) { return (nq >= 8 || nq < 0) ? 1 : 4; }
__host__ __device__ inline size_t emit_slab_bytes(int Lp) { return ((size_t)2 * Lp * sizeof(int) + 127) / 128 * 128; }
__host__ __device__ inline size_t emit_smem_bytes(int Lp, int staged_V) {
    return staged_V ? emit_slab_bytes(Lp) + (size_t)kG * staged_V * 4 + 64 : (size_t)2 * Lp * sizeof(int);
}

// DEC (loss evaluation with the greedy decode, ctcb_forward_decode_typed): every valid frame's best two symbols from the
// values the variant already holds, one word per frame into dec.tok (decode_word); dec is read by these variants only
template <int VEC, int NQ, typename LT = float, bool DEC = false>
__global__ void __launch_bounds__(NQ < 0 ? 256 : 128) k_emit(Problem p, Workspace w, DecodeOut dec) {
    using V_t = typename LV<LT, VEC>::type;
    using S_t = typename LV<LT, 4>::type;          // staged rows: four elements per shared-memory load
    // (a programmatic dependent -- the fused projection, ctcb_proj.cuh -- needs nothing from this kernel and may start at once)
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    extern __shared__ __align__(128) int slab[];  // 2*Lp ints: this utterance's labels, metadata scratch
    __shared__ int s_L, s_rep, s_flags;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr bool STAGED = NQ < 0;
    const int b = blockIdx.y;
    const int xi = (int)blockIdx.x;
    constexpr int NT = STAGED ? 256 : 128;        // staged rows: 8 warps, one row each
    float* srow = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(slab) + emit_slab_bytes(w.Lp));   // kG rows of V floats
    uint64_t* rbar = reinterpret_cast<uint64_t*>(srow + (size_t)kG * p.V);
    LT* srowL = reinterpret_cast<LT*>(srow);      // row j at element j * V (bf16 rows fill the first half of the area)
    if (tid == 0) { s_L = p.Lmax; s_rep = 0; s_flags = 0; }
    __syncthreads();
    // operator parameter layer: lengths (trunc + clamp) and labels (trunc + clamp)
    int Tb = p.T, lenflags = 0;
    if (p.data_len) {
        long long t64 = load_as_int(p.data_len, p.data_len_dtype, b);
        if (t64 < 0) { t64 = 0; lenflags = UTT_LEN_CLAMPED; }
        if (t64 > p.T) { t64 = p.T; lenflags = UTT_LEN_CLAMPED; }
        Tb = (int)t64;
    }
    int L;
    if (p.label_len) {
        long long l64 = load_as_int(p.label_len, p.label_len_dtype, b);
        if (l64 < 0) { l64 = 0; lenflags = UTT_LEN_CLAMPED; }
        if (l64 > p.Lmax) { l64 = p.Lmax; lenflags = UTT_LEN_CLAMPED; }
        L = (int)l64;
    } else {
        for (int j = tid; j < p.Lmax; j += NT)
            if (load_as_int(p.labels, p.label_dtype, b * p.lst_b + j * p.lst_l) == p.label_pad) atomicMin(&s_L, j);
        __syncthreads();
        L = s_L;
    }
    const bool meta_cta = blockIdx.x == gridDim.x - 1;       // one extra CTA per utterance: metadata only
    const int sblk = xi;
    if (STAGED && !meta_cta && lane == 0 && sblk * kG < Tb) {
        // this warp's row: requested before anything else, consumed below
        const int t = sblk * kG + warp;
        mbar_init(rbar + warp, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (t < Tb) {
            mbar_expect_tx(rbar + warp, (uint32_t)p.V * (uint32_t)sizeof(LT));
            tma_load_1d(srowL + (size_t)warp * p.V, utt_logits<LT>(p, b) + (long long)t * p.st_t, (uint32_t)p.V * (uint32_t)sizeof(LT), rbar + warp);
        }
    }
    __syncwarp();
    if (!w.dense || meta_cta) {
        int bad = 0;
        for (int j = tid; j < L; j += NT) {
            long long v = load_as_int(p.labels, p.label_dtype, b * p.lst_b + j * p.lst_l);
            if (v < 0 || v >= p.V || v == p.blank) bad = 1;
            slab[j] = (int)(v < 0 ? 0 : (v >= p.V ? p.V - 1 : v));
        }
        if (bad) atomicOr(&s_flags, UTT_BAD_LABEL);
        __syncthreads();
    }

    const int nvec = p.V / VEC;
    // frame blocks per CTA: one warp per block, or -- for wide rows (8 or 16 vector loads per lane) --
    // one block per CTA with two frames per warp: four times as many CTAs, so the grid is several
    // waves deep and every SM keeps more row loads in flight
    constexpr int BPC = emit_blocks_per_cta(NQ), FPW = kG * BPC / 4;
    const int blk = BPC == 4 ? blockIdx.x * 4 + warp : (STAGED ? sblk : (int)blockIdx.x), t0 = blk * kG;
    const int jbeg = BPC == 4 ? 0 : warp * FPW;
    if (!meta_cta && t0 < Tb) {
        float mxs[kG];
        const LT* rows = utt_logits<LT>(p, b) + (long long)t0 * p.st_t;
        if (STAGED) {
            __shared__ float s_mx[kG];
            if (t0 + warp < Tb) {
                mbar_wait(rbar + warp, 0);
                const S_t* sv = reinterpret_cast<const S_t*>(srowL + (size_t)warp * p.V);
                float m0 = -INFINITY, m1 = -INFINITY;
                Top2 tp = kTop2Empty;
                for (int k = lane; k < nvec; k += 64) {
                    float a[4]; LV<LT, 4>::get(sv[k], a);
                    m0 = fmaxf(m0, fmaxf(fmaxf(a[0], a[1]), fmaxf(a[2], a[3])));
                    if (DEC) {
#pragma unroll
                        for (int i = 0; i < 4; ++i) top2_insert(tp, a[i], 4 * k + i);
                    }
                    if (k + 32 < nvec) {
                        float c[4]; LV<LT, 4>::get(sv[k + 32], c); m1 = fmaxf(m1, fmaxf(fmaxf(c[0], c[1]), fmaxf(c[2], c[3])));
                        if (DEC) {
#pragma unroll
                            for (int i = 0; i < 4; ++i) top2_insert(tp, c[i], 4 * (k + 32) + i);
                        }
                    }
                }
                const float mx = warp_max(fmaxf(m0, m1));
                if (DEC) {
                    top2_warp_merge(tp, dec.unk >= 0);
                    if (lane == 0) dec.tok[(size_t)b * p.T + t0 + warp] = decode_word(tp, dec.unk);
                }
                float s0 = 0.0f, s1 = 0.0f;
                for (int k = lane; k < nvec; k += 64) {
                    float a[4]; LV<LT, 4>::get(sv[k], a);
                    s0 += fast_ex2((a[0] - mx) * kLog2e) + fast_ex2((a[1] - mx) * kLog2e);
                    s1 += fast_ex2((a[2] - mx) * kLog2e) + fast_ex2((a[3] - mx) * kLog2e);
                    if (k + 32 < nvec) {
                        float c[4]; LV<LT, 4>::get(sv[k + 32], c);
                        s0 += fast_ex2((c[0] - mx) * kLog2e) + fast_ex2((c[1] - mx) * kLog2e);
                        s1 += fast_ex2((c[2] - mx) * kLog2e) + fast_ex2((c[3] - mx) * kLog2e);
                    }
                }
                const float sum = warp_sum(s0 + s1);
                if (lane == 0) { w.fr[(size_t)b * p.T + t0 + warp] = make_float2(mx, log2f(sum)); s_mx[warp] = mx; }
            } else if (lane == 0) s_mx[warp] = 0.0f;
            __syncthreads();
            // the emission columns of the block's 8 frames, gathered from the staged rows: one thread per column,
            // 64 contiguous bytes each
            const int ncol = w.dense ? p.V : L + 1;
            const int nval = min(kG, Tb - t0);
            double* eblk = w.E + ((size_t)b * w.NB + blk) * w.W * kEC;
            bool floored = false;
            for (int col = tid; col < ncol; col += NT) {
                const int v = w.dense ? col : (col == 0 ? p.blank : slab[col - 1]);
                double y[kG];
#pragma unroll
                for (int j = 0; j < kG; ++j) {
                    const float l2 = (ldsx(srowL + (size_t)j * p.V + v) - s_mx[j]) * kLog2e;
                    floored |= j < nval && l2 < kMinLog2;
                    y[j] = j < nval ? (double)fast_ex2(fmaxf(l2, kMinLog2)) : 0.0;
                }
                double2* dst = reinterpret_cast<double2*>(eblk + (size_t)col * kEC);
#pragma unroll
                for (int j = 0; j < kG; j += 2) dst[j / 2] = make_double2(y[j], y[j + 1]);
            }
            if (floored && p.status) atomicOr(p.status + b, UTT_WIDE_LOGITS);
        } else if (NQ > 0) {
            constexpr int NQ1 = NQ > 0 ? NQ : 1;
            constexpr int F = NQ1 >= 16 ? 1 : (NQ1 >= 8 ? 2 : (NQ1 >= 4 ? 4 : 8));
#pragma unroll
            for (int jk = 0; jk < FPW; jk += F) {
                const int jf = jbeg + jk;
                V_t x[F][NQ1]; float xt[F];
#pragma unroll
                for (int f = 0; f < F; ++f) {                   // every load of F frames in flight
                    const bool valid = t0 + jf + f < Tb;
                    const LT* row = rows + (jf + f) * p.st_t;
                    const V_t* rowv = reinterpret_cast<const V_t*>(row);
#pragma unroll
                    for (int q = 0; q < NQ1; ++q) {
                        const int k = q * 32 + lane;
                        x[f][q] = (valid && k < nvec) ? __ldg(rowv + k) : LV<LT, VEC>::fill(-INFINITY);
                    }
                    xt[f] = (VEC > 1 && valid && nvec * VEC + lane < p.V) ? ldx(row + nvec * VEC + lane) : -INFINITY;
                }
                float mx[F], sum[F];
#pragma unroll
                for (int f = 0; f < F; ++f) {
                    float m = xt[f];
#pragma unroll
                    for (int q = 0; q < NQ1; ++q) { float e[VEC]; LV<LT, VEC>::get(x[f][q], e);
#pragma unroll
                        for (int i = 0; i < VEC; ++i) m = fmaxf(m, e[i]); }
                    mx[f] = m;
                }
                if (DEC) {
                    // frame by frame: the lane's columns (tail included), the warp's merge, lane f writes frame f's word
#pragma unroll
                    for (int f = 0; f < F; ++f) {
                        Top2 tp = kTop2Empty;
                        if (VEC > 1 && nvec * VEC + lane < p.V) top2_insert(tp, xt[f], nvec * VEC + lane);
#pragma unroll
                        for (int q = 0; q < NQ1; ++q) {
                            if (q * 32 + lane >= nvec) continue;         // the -inf fill of absent loads is not a column
                            float e[VEC]; LV<LT, VEC>::get(x[f][q], e);
#pragma unroll
                            for (int i = 0; i < VEC; ++i) top2_insert(tp, e[i], (q * 32 + lane) * VEC + i);
                        }
                        top2_warp_merge(tp, dec.unk >= 0);
                        if (lane == f && t0 + jf + f < Tb) dec.tok[(size_t)b * p.T + t0 + jf + f] = decode_word(tp, dec.unk);
                    }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1)
#pragma unroll
                    for (int f = 0; f < F; ++f) mx[f] = fmaxf(mx[f], __shfl_xor_sync(0xffffffffu, mx[f], o));
#pragma unroll
                for (int f = 0; f < F; ++f) {
                    float sacc = fast_ex2((xt[f] - mx[f]) * kLog2e);          // ex2(-inf) = 0 for absent elements
#pragma unroll
                    for (int q = 0; q < NQ1; ++q) { float e[VEC]; LV<LT, VEC>::get(x[f][q], e);
#pragma unroll
                        for (int i = 0; i < VEC; ++i) sacc += fast_ex2((e[i] - mx[f]) * kLog2e); }
                    sum[f] = sacc;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1)
#pragma unroll
                    for (int f = 0; f < F; ++f) sum[f] += __shfl_xor_sync(0xffffffffu, sum[f], o);
#pragma unroll
                for (int f = 0; f < F; ++f) {
                    mxs[jf + f] = mx[f];
                    if (lane == f && t0 + jf + f < Tb) w.fr[(size_t)b * p.T + t0 + jf + f] = make_float2(mx[f], log2f(sum[f]));
                }
                // the emission columns of these frames NOW, while their rows are still in L1: gathering
                // after the whole block re-read evicted rows from L2/HBM (ncu: 1.26x the compulsory bytes)
                {
                    const int ncol = w.dense ? p.V : L + 1;
                    double* eblk = w.E + ((size_t)b * w.NB + blk) * w.W * kEC;
                    for (int col = lane; col < ncol; col += 32) {
                        const int v = w.dense ? col : (col == 0 ? p.blank : slab[col - 1]);
#pragma unroll
                        for (int f = 0; f < F; ++f) {
                            const bool valid = t0 + jf + f < Tb;
                            const float xv = valid ? ldx(rows + (jf + f) * p.st_t + v) : 0.0f;
                            if (valid && (xv - mx[f]) * kLog2e < kMinLog2 && p.status) atomicOr(p.status + b, UTT_WIDE_LOGITS);
                            eblk[(size_t)col * kEC + jf + f] = valid ? (double)fast_ex2(fmaxf((xv - mx[f]) * kLog2e, kMinLog2)) : 0.0;
                        }
                    }
                }
            }
        } else {
#pragma unroll
            for (int j = 0; j < kG; ++j) {
                const int t = t0 + j;
                mxs[j] = 0.0f;
                if (t >= Tb) continue;
                const LT* row = rows + j * p.st_t;
                const V_t* rowv = reinterpret_cast<const V_t*>(row);
                float mx = -INFINITY;
                Top2 tp = kTop2Empty;
                for (int k = lane; k < nvec; k += 32) {
                    float x[VEC]; LV<LT, VEC>::get(__ldg(rowv + k), x);
#pragma unroll
                    for (int i = 0; i < VEC; ++i) { mx = fmaxf(mx, x[i]); if (DEC) top2_insert(tp, x[i], k * VEC + i); }
                }
                for (int v = nvec * VEC + lane; v < p.V; v += 32) {
                    const float xv = ldx(row + v);
                    mx = fmaxf(mx, xv);
                    if (DEC) top2_insert(tp, xv, v);
                }
                mx = warp_max(mx);
                if (DEC) {
                    top2_warp_merge(tp, dec.unk >= 0);
                    if (lane == 0) dec.tok[(size_t)b * p.T + t] = decode_word(tp, dec.unk);
                }
                float sum = 0.0f;
                for (int k = lane; k < nvec; k += 32) {          // second pass hits L1/L2
                    float x[VEC]; LV<LT, VEC>::get(__ldg(rowv + k), x);
#pragma unroll
                    for (int i = 0; i < VEC; ++i) sum += fast_ex2((x[i] - mx) * kLog2e);
                }
                for (int v = nvec * VEC + lane; v < p.V; v += 32) sum += fast_ex2((ldx(row + v) - mx) * kLog2e);
                sum = warp_sum(sum);
                if (lane == 0) w.fr[(size_t)b * p.T + t] = make_float2(mx, log2f(sum));
                mxs[j] = mx;
            }
        }
        const int ncol = NQ != 0 ? 0 : (w.dense ? p.V : L + 1);     // NQ != 0: already written frame by frame
        double* eblk = w.E + ((size_t)b * w.NB + blk) * w.W * kEC;
        for (int col = lane; col < ncol; col += 32) {
            const int v = w.dense ? col : (col == 0 ? p.blank : slab[col - 1]);
            float xv[kG];
#pragma unroll
            for (int j = 0; j < kG; ++j) xv[j] = t0 + j < Tb ? ldx(rows + j * p.st_t + v) : 0.0f;
            double2* dst = reinterpret_cast<double2*>(eblk + (size_t)col * kEC);
#pragma unroll
            for (int j = 0; j < kG; j += 2) {
                const double y0 = t0 + j < Tb ? (double)fast_ex2(fmaxf((xv[j] - mxs[j]) * kLog2e, kMinLog2)) : 0.0;
                const double y1 = t0 + j + 1 < Tb ? (double)fast_ex2(fmaxf((xv[j + 1] - mxs[j + 1]) * kLog2e, kMinLog2)) : 0.0;
                if (p.status && ((t0 + j < Tb && (xv[j] - mxs[j]) * kLog2e < kMinLog2) ||
                                 (t0 + j + 1 < Tb && (xv[j + 1] - mxs[j + 1]) * kLog2e < kMinLog2)))
                    atomicOr(p.status + b, UTT_WIDE_LOGITS);
                dst[j / 2] = make_double2(y0, y1);
            }
        }
    }

    if (!meta_cta) return;
    // ---- per-utterance metadata ----
    // The gradient kernel sums the occupancy of every occurrence of a label value into that
    // value's column in a FIXED order (no atomics): it writes the occupancies at their rank in
    // the order (value, position), so that each distinct value is one contiguous run, and walks the
    // list of distinct values {value, start of its run}.  Ranks by counting (L <= 2047).
    int* lab = w.lab + (size_t)b * w.Lp;
    int* rank = w.rank + (size_t)b * w.Lp;
    int2* dl = w.dl + (size_t)b * (w.Lp + 1);
    int* s_run = slab + w.Lp;                      // start of the run a position opens, or -1
    __shared__ int s_nd;
    if (tid == 0) s_nd = 0;
    int rep = 0;
    for (int j = tid; j < L; j += NT) {
        const int v = slab[j];
        lab[j] = v;
        if (j > 0 && slab[j - 1] == v) ++rep;
        int lt = 0, eqb = 0;
        for (int k = 0; k < L; ++k) { const int u = slab[k]; lt += u < v; eqb += (u == v) & (k < j); }
        rank[j] = lt + eqb;
        s_run[j] = eqb == 0 ? lt : -1;
    }
    if (rep) atomicAdd(&s_rep, rep);
    __syncthreads();
    int mine = 0;
    for (int j = tid; j < L; j += NT) {
        if (s_run[j] < 0) continue;
        const int v = slab[j];
        int d = 0;
        for (int k = 0; k < L; ++k) d += (s_run[k] >= 0) & (slab[k] < v);
        dl[d] = make_int2(v, s_run[j]);
        ++mine;
    }
    if (mine) atomicAdd(&s_nd, mine);
    __syncthreads();
    if (tid == 0) {
        int flags = s_flags | lenflags;
        if (Tb <= 0 || L + s_rep > Tb) flags |= UTT_INFEASIBLE;
        w.Tb[b] = Tb; w.Lb[b] = L; w.flags[b] = flags;
        w.nd[b] = s_nd; dl[s_nd] = make_int2(-1, L);
        if (p.status && flags) atomicOr(p.status + b, flags);   // zeroed by the host before the call; frame CTAs OR their bits in
        if (flags & UTT_INFEASIBLE) p.loss[b] = 0.0f;   // defined behaviour, SURVEY 7.3-6
        w.gprog[4 * b] = 0; w.gprog[4 * b + 1] = 0; w.gprog[4 * b + 3] = 0;
        __threadfence();
        st_release_gpu(w.gprog + 4 * b + 2, w.stamp);      // "metadata ready": a recursion kernel that runs beside this one polls it
    }
}

// ---------------------------------------------------------------------------------------
// mbarrier / TMA (1-D bulk copy) / shared-memory helpers
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "W_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra D_%=;\n\t"
        "bra W_%=;\n\t"
        "D_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// wait of a warp that has slack (producers run many blocks ahead): it shares an SM sub-partition
// with a walker warp whose dependent chain is the critical path, so it must not spin on the issue port
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity, int hw_wait = 0) {
    // hw_wait: mbarrier.try_wait suspends the warp in hardware -- no polling instructions at all, which is what
    // counts when several walker CTAs share an SM and the kernel is bound by instruction issue (throughput
    // regime: the nanosleep polls were a quarter of k_walk's executed instructions at B = 1024)
    if (hw_wait) { mbar_wait(bar, parity); return; }
    while (!mbar_test(bar, parity)) __nanosleep(128);
}
__device__ __forceinline__ void st_release_gpu(int* p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
    int v; asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v;
}
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// shared -> global bulk copy (asynchronous proxy): the row was written with ordinary stores, hence the proxy fence
__device__ __forceinline__ void tma_store_1d(void* dst_gmem, const void* src_smem, uint32_t bytes) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void tma_store_wait_read() {   // the source rows may be reused / the CTA may exit
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ double lds_f64(uint32_t addr) {
    double v; asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr)); return v;
}
__device__ __forceinline__ void sts_f64(uint32_t addr, double v) {
    asm volatile("st.shared.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory");
}
__device__ __forceinline__ int lds_acquire(uint32_t addr) {
    int v; asm volatile("ld.acquire.cta.shared.s32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory"); return v;
}
__device__ __forceinline__ void sts_release(uint32_t addr, int v) {
    asm volatile("st.release.cta.shared.s32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ int lds_relaxed(uint32_t addr) {
    int v; asm volatile("ld.relaxed.cta.shared.s32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory"); return v;
}
__device__ __forceinline__ void sts_s32(uint32_t addr, int v) {
    asm volatile("st.shared.s32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

__device__ __forceinline__ double2 lds_v2f64(uint32_t addr) {
    double2 v; asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr)); return v;
}

// ---------------------------------------------------------------------------------------
// k_walk<P,NW,HIST>: grid (B, ndir), block (NW+1)*32.  Rows a6/a7 (the two recursions).
//
// Slot g (= walker thread * P + p) owns the state pair (blank 2g, label 2g+1) of the walker's
// lattice.  dir 0 walks frames 0..T_b-1 over ext = [_, l1, _, ..., lL, _] and stores alpha_t
// (emission included); dir 1 walks frames T_b-1..0 over the REVERSED label sequence -- which
// is exactly the beta recursion -- and stores the sum BEFORE the emission is applied
// (beta'_t), so that  sum_s alpha_t(s) beta'_t(S-1-s) = P(l|x)  for every t.
//
// Number format.  A state's value is  v * 2^e : v an fp64 held in a register, e an int32
// "offset" that is constant between renormalisations.  One step is, per pair,
//     sb = prev*fb + b          sl = prev*fls + (b*flb + l)        b' = sb*y_blank   l' = sl*y_label
// (5 FP64 ops) where prev is the neighbouring label state (warp shuffle) and fb, fls, flb are
// the cached powers of two 2^(e_source - e_destination) (fls = 0 where the skip transition is
// not allowed).  Emissions are in [2^-100, 1], so in one group of kG = 8 steps a value
// shrinks by at most 2^-800 and grows by at most 3^8 * 2^(8 kD): it cannot leave the fp64
// range when it starts a group within 2^+-kDrift of its offset.  At a group boundary a warp
// renormalises only if some state drifted past 2^+-kDrift or its left neighbour's offsets
// changed; otherwise the boundary costs one vote.  Renormalising moves every state's exponent
// into its offset; if there are exactly-zero states (beyond the wavefront) or neighbouring
// offsets more than 2^kD apart, a max-plus scan with decay kD per pair keeps every cached
// factor <= 2^kD and gives the zero states the offset of the front.
// States beyond the utterance's lattice are not masked: probability only flows towards higher
// states, so whatever they hold never reaches a valid state, the loss or the stored history.
//
// Execution: NW walker warps + 1 producer warp; the step loop has NO CTA barrier.
//   * producer warp: streams E frame blocks (kG frames, frame-minor) into a shared-memory ring
//     with cp.async.bulk (TMA) + full/empty mbarriers; the alpha CTA's producer also sums
//     log2(softmax denominator) over the utterance's frames for the loss;
//   * walkers take a whole block of emissions into registers with 128-bit shared loads, run
//     its 8 steps fully unrolled, and store the history with immediate offsets into the
//     block's per-warp chunk;
//   * walker warp w needs, per step, one value from warp w-1 (its last label state at the
//     previous step).  Warp w-1 stores it into a 4-group-deep ring and, after each group,
//     publishes its group count (release); warp w starts group j once warp w-1 has finished
//     group j (acquire).  Warps therefore run as a wavefront skewed by one group, each at the
//     speed of its own dependent chain.  Per group each warp also publishes {last label state,
//     its offset, scan carry, front offset} for its right neighbour.
// The beta walker's groups are aligned to the same frame blocks (its first group is the
// partial one), so both histories and both offset tables are indexed by t / 8.
// ---------------------------------------------------------------------------------------
struct WalkArgs {
    Problem p;             // read by the fused variant only (parameter layer + logits)
    Workspace w; int T; int stages; int blank; float* loss; double* loss_sum;
    long long* trace;      // debug only (scripts/ubench/walk_trace.cu); nullptr in the product
    int hw_wait;           // producers wait on mbarrier.try_wait (hardware suspend) instead of nanosleep polls
    int publish;           // 1: the progress of every group is published promptly (gradient CTAs run concurrently);
                           // 2: lazily (the gradient kernel runs after this one: only the final count matters)
    int meet;              // loss evaluation only (no history): the alpha walker takes the first half of the frame blocks, the
                           // beta walker the second half from the end, and P(l|x) = sum_s alpha_m(s) beta'_m(s) is formed
                           // at the meeting frame by whichever warp hands over last -- half the dependent chain
    int pdl_wait;          // launched with programmatic stream serialization behind an arbitrary kernel (the previous step's
                           // gradient kernel, a model's last kernel): the CTAs become resident during that kernel's tail
                           // and execute griddepcontrol.wait before they touch memory
    int beside_proj;       // unfused variant launched as the programmatic dependent of the fused projection: metadata and
                           // emission blocks are awaited through Workspace::gprog / tflag instead of the stream order
    DecodeOut dec;         // read by the decoding variant only (k_walk's DEC): where its producers leave each frame's word
};

#ifdef CTCB_TRACE
#define CTCB_TP(id) do { if (a.trace && blockIdx.x == 0 && lane == 0) \
    a.trace[((size_t)(blockIdx.y * 32 + warp) * 4096 + (size_t)n * 8 + (id))] = clock64(); } while (0)
#else
#define CTCB_TP(id) do { } while (0)
#endif

struct HaloMeta { double lm; int el; int R; int F; int pad; };   // 24 bytes, 8-byte aligned
constexpr int kHaloDepth = 16;   // halo ring depth in groups (= kMaxStages): a warp cannot lead its right neighbour by more
                                 // than the emission ring holds, because a ring stage is recycled only when every warp is done with it

constexpr int kFusedProducers = 2;      // fused variant: warps that turn logits rows into emission blocks

// fused_Lp > 0: the fused variant also keeps the utterance's int labels (fused_Lp ints)
__host__ __device__ inline size_t walk_smem_bytes(int W, int NW, int stages, int fused_Lp = 0) {
    return (size_t)stages * kEC * W * sizeof(double) + 2 * kMaxStages * sizeof(uint64_t) +
           (size_t)NW * kHaloDepth * kG * sizeof(double) + (size_t)NW * kHaloDepth * sizeof(HaloMeta) +
           (size_t)NW * sizeof(int) + 64 + (fused_Lp ? 16 + kFusedProducers * 64 + (size_t)fused_Lp * sizeof(int) : 0);
}

template <int P, int NW, int DIR, bool HIST, bool FUSED, typename LT = float, bool DEC = false>
__device__ __forceinline__ void walk_dir(const WalkArgs& a, unsigned char* smem_raw, int Tb, int Lb, int uflags) {
    constexpr int PW = 32 * P;
    constexpr unsigned FULL = 0xffffffffu;
    const Workspace& w = a.w;
    const int b = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int W = w.W, NS = a.stages;
    const int NQ = (Tb + kG - 1) / kG;              // frame blocks of this utterance
    const int rlast = Tb - (NQ - 1) * kG;           // frames in the last block, 1..8
    // meeting in the middle (loss evaluation): alpha walks blocks [0, Mblk), beta blocks [Mblk, NQ) from the end
    const bool meet = !HIST && a.meet && NQ >= 2;
    const int Mblk = (NQ + 1) / 2;
    const int NQr = meet ? (DIR ? NQ - Mblk : Mblk) : NQ;      // groups this walker runs
    if (!HIST && DIR == 1 && !meet) return;         // an utterance too short to split: the alpha CTA does it all
    const uint32_t stage_bytes = (uint32_t)W * kEC * 8u;

    const uint32_t ring = smem_u32(smem_raw);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)NS * stage_bytes);
    uint64_t* empty = full + kMaxStages;
    const uint32_t halo = smem_u32(empty + kMaxStages);                          // [NW][4][kG] double
    const uint32_t meta = halo + NW * kHaloDepth * kG * 8;                       // [NW][4] HaloMeta
    const uint32_t prog = meta + NW * kHaloDepth * (uint32_t)sizeof(HaloMeta);   // [NW] int: groups completed
    const uint32_t lsum = (prog + NW * 4 + 7u) & ~7u;      // double + int flag; fused: 8 doubles per producer warp at +16
    int* slab = reinterpret_cast<int*>(smem_raw + (lsum - ring) + 32 + kFusedProducers * 64);           // fused: Lp int labels (filled by k_walk)

    if (tid == 0) {
        for (int s = 0; s < NS; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], NW); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        sts_s32(lsum + 8, 0);
        if (FUSED) for (int q = 0; q < kFusedProducers * 8; ++q) sts_f64(lsum + 16 + q * 8, 0.0);
    }
    if (tid < NW) sts_s32(prog + tid * 4, 0);
    __syncthreads();

    if (FUSED && warp >= NW && warp < NW + kFusedProducers) {
        // ---- fused producer warps: logits rows -> emission blocks, straight into the ring ----
        // Producer q owns the walker groups n = q, q + 2, ...  Four lanes share one frame of the
        // block (lane = 4*frame + quarter), each holding a contiguous quarter of the row (<= 16
        // columns, V <= 64, any stride or alignment): row max and sum need two shuffle steps per
        // block instead of a full warp reduction per frame -- the walkers' own shuffles, which sit
        // on the critical path, go through the same SM-wide pipe.  Every load of the NEXT block is
        // in flight while this one is reduced.  The alpha CTA also keeps {row max, log2 sum} per
        // frame for the gradient's softmax and sums log2(sum) for the loss.
        const Problem& p = a.p;
        constexpr int CPL = 16;                                        // columns per lane, at most
        const int q = warp - NW, V = p.V;
        const int fj = lane >> 2, qk = lane & 3;                       // frame of the block, quarter of the row
        const int cpl = (V + 3) >> 2, col0 = qk * cpl;                 // this lane's columns [col0, col0 + cpl) below V
        const LT* base = utt_logits<LT>(p, b);
        const float kMinProb = 7.888609052210118e-31f;                 // 2^kMinLog2
        auto load_blk = [&](int n, float (&x)[CPL]) {
            const int t = (DIR ? NQ - 1 - n : n) * kG + fj;
            const LT* row = base + (long long)t * p.st_t + col0;
            const bool valid = t < Tb;
#pragma unroll
            for (int i = 0; i < CPL; ++i) x[i] = (valid && i < cpl && col0 + i < V) ? ldx(row + i) : -INFINITY;
        };
        float cur[CPL], nxt[CPL];
        double ls = 0.0;
        bool floored = false;
        int n = q;
        if (n < NQr) load_blk(n, cur);
#pragma unroll 1
        for (; n < NQr; n += kFusedProducers) {
            if (n + kFusedProducers < NQr) load_blk(n + kFusedProducers, nxt);
            const int t = (DIR ? NQ - 1 - n : n) * kG + fj;
            const bool valid = t < Tb;
            float mx = cur[0];
#pragma unroll
            for (int i = 1; i < CPL; ++i) mx = fmaxf(mx, cur[i]);
            mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, 1));
            mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, 2));
            if (DEC) {
                // the greedy decode while the row is in registers: each frame's best two of its four lanes' columns
                // (two shuffle steps; the best alone without an <unk> rule), one word per valid frame.  The alpha
                // producers cover blocks [0, NQr), the beta producers under `meet` the others: every valid frame once
                Top2 tp = kTop2Empty;
#pragma unroll
                for (int i = 0; i < CPL; ++i)
                    if (i < cpl && col0 + i < V) top2_insert(tp, cur[i], col0 + i);
                const bool two = a.dec.unk >= 0;
                top2_merge_xor(tp, 1, two);
                top2_merge_xor(tp, 2, two);
                if (valid && qk == 0) a.dec.tok[(size_t)b * a.T + t] = decode_word(tp, a.dec.unk);
            }
            float e[CPL], sm = 0.0f;
#pragma unroll
            for (int i = 0; i < CPL; ++i) {                            // rows past T_b are all -inf: keep NaN out
                e[i] = valid ? fast_ex2((cur[i] - mx) * kLog2e) : 0.0f;
                sm += e[i];
                // an emission below the floor (any symbol of a valid frame): reported, UTT_WIDE_LOGITS
                if (DIR == 0 || meet) floored |= valid && i < cpl && col0 + i < V && e[i] < kMinProb;
            }
            sm += __shfl_xor_sync(FULL, sm, 1);
            sm += __shfl_xor_sync(FULL, sm, 2);
            if ((DIR == 0 || meet) && valid && qk == 0) {
                const float l2 = log2f(sm);
                ls += (double)l2;
                if (DIR == 0) w.fr[(size_t)b * a.T + t] = make_float2(mx, l2);
            }
            const int st = n % NS, use = n / NS;
            if (use > 0) mbar_wait_relaxed(&empty[st], (uint32_t)((use - 1) & 1), a.hw_wait);
            const uint32_t dst = ring + (uint32_t)st * stage_bytes + (uint32_t)col0 * (kEC * 8u) + (uint32_t)fj * 8u;
#pragma unroll
            for (int i = 0; i < CPL; ++i)
                if (i < cpl && col0 + i < V) sts_f64(dst + (uint32_t)i * (kEC * 8u), valid ? (double)fmaxf(e[i], kMinProb) : 0.0);
            if ((DIR == 0 || meet) && qk == 0) sts_f64(lsum + 16 + (q * 8 + fj) * 8, ls);   // before the arrive: the walkers' acquire covers it
            __syncwarp();
            if (lane == 0) mbar_arrive(&full[st]);
#pragma unroll
            for (int i = 0; i < CPL; ++i) cur[i] = nxt[i];
        }
        if ((DIR == 0 || meet) && p.status && __any_sync(FULL, floored) && lane == 0) atomicOr(p.status + b, UTT_WIDE_LOGITS);
        return;
    }
    if (FUSED && warp == NW + kFusedProducers) {
        // ---- fused publisher warp ----
        const Problem& p = a.p;
        if (DIR == 0 && HIST) {
            // metadata of the gradient kernel (what k_emit's extra CTA writes in the unfused path); the
            // vocabulary has at most 64 symbols, so ranks come from two counting passes over the labels
            int* rank = w.rank + (size_t)b * w.Lp;
            int2* dl = w.dl + (size_t)b * (w.Lp + 1);
            int c0 = 0, c1 = 0;
            for (int j = 0; j < Lb; ++j) { const int v = slab[j]; c0 += v == lane; c1 += v == lane + 32; }
            int i0 = c0, i1 = c1;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y0 = __shfl_up_sync(FULL, i0, o), y1 = __shfl_up_sync(FULL, i1, o);
                if (lane >= o) { i0 += y0; i1 += y1; }
            }
            const int tot0 = __shfl_sync(FULL, i0, 31);
            int r0 = i0 - c0, r1 = tot0 + i1 - c1;
            const unsigned m0 = __ballot_sync(FULL, c0 > 0), m1 = __ballot_sync(FULL, c1 > 0);
            const unsigned below = (1u << lane) - 1u;
            const int nd = __popc(m0) + __popc(m1);
            if (c0 > 0) dl[__popc(m0 & below)] = make_int2(lane, r0);
            if (c1 > 0) dl[__popc(m0) + __popc(m1 & below)] = make_int2(lane + 32, r1);
            w.runv[(size_t)b * 64 + lane] = make_int2(r0, r0 + c0);
            w.runv[(size_t)b * 64 + lane + 32] = make_int2(r1, r1 + c1);
            for (int j = 0; j < Lb; ++j) {
                const int v = slab[j];
                if (v == lane) rank[j] = r0++;
                else if (v == lane + 32) rank[j] = r1++;
            }
            if (lane == 0) {
                dl[nd] = make_int2(-1, Lb);
                w.nd[b] = nd; w.Tb[b] = Tb; w.Lb[b] = Lb; w.flags[b] = uflags;
            }
            __syncwarp();
            if (lane == 0) st_release_gpu(w.gprog + 4 * b + 2, w.stamp);
        }
        if (HIST && lane == 0 && a.publish) {
            // the last walker warp's group count (shared memory) -> global progress for the gradient CTAs
            int* gp = w.gprog + 4 * b + DIR;
            const uint32_t last_prog = prog + (NW - 1) * 4;
            int seen = 0;
            while (seen < NQ) {
                const int v = lds_acquire(last_prog);
                if (v > seen) { st_release_gpu(gp, v); seen = v; }
                else __nanosleep(a.publish == 2 ? 4000 : 128);
            }
        }
        (void)p;
        return;
    }

    if (!FUSED && warp == NW) {                 // ---- producer warp (emission table from k_emit, by TMA) ----
        const double* Eb = w.E + (size_t)b * w.NB * W * kEC;
        int tile_seen = -1;                     // beside the projection: the last 128-frame tile known to be written
        auto issue = [&](int n, int st) {       // block of walker group n into ring stage st
            const int blk = DIR ? NQ - 1 - n : n;
            if (a.beside_proj && (blk >> 4) != tile_seen) {
                const int* f = w.tflag + (size_t)b * w.ntile + (blk >> 4);
                const long long t0 = clock64();     // bounded: a projection that never ran gives garbage, not a hang
                while (ld_acquire_gpu(f) == 0 && clock64() - t0 < kSpinLimit) __nanosleep(256);
                asm volatile("fence.proxy.async;" ::: "memory");     // the bulk copy below reads what generic stores wrote
                tile_seen = blk >> 4;
            }
            mbar_expect_tx(&full[st], stage_bytes);
            tma_load_1d(smem_raw + (size_t)st * stage_bytes, Eb + (size_t)blk * W * kEC, stage_bytes, &full[st]);
        };
        const int npro = min(NS, NQr);
        if (lane == 0) for (int n = 0; n < npro; ++n) issue(n, n);
        // this walker's frames: all of them, or its side of the meeting frame
        const int t_lo = (meet && DIR) ? Mblk * kG : 0, t_hi = (meet && !DIR) ? min(Tb, Mblk * kG) : Tb;
        if ((DIR == 0 || meet) && !a.beside_proj) {       // sum_t log2(softmax denominator), fixed order
            double s = 0.0;
            for (int t = t_lo + lane; t < t_hi; t += 32) s += (double)w.fr[(size_t)b * a.T + t].y;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                s += __hiloint2double(__shfl_xor_sync(FULL, __double2hiint(s), o), __shfl_xor_sync(FULL, __double2loint(s), o));
            }
            if (lane == 0) { sts_f64(lsum, s); sts_release(lsum + 8, 1); }
        }
        if (lane == 0) {
            // Group n is complete (every walker warp handed its ring stage back, after storing its
            // history) -> refill the stage with block n + NS and publish the progress for the
            // gradient CTAs, which run concurrently (k_grad is a programmatic dependent of this
            // kernel).  A completion that is immediately followed by the next one is not published
            // on its own: the fence of a release at gpu scope costs about one group.
            int* gp = HIST ? w.gprog + 4 * b + DIR : nullptr;
            int st = 0; uint32_t par = 0;
            for (int n = 0; n < NQr; ++n) {
                mbar_wait_relaxed(&empty[st], par, a.hw_wait);
                if (n + NS < NQr) issue(n + NS, st);
                if (++st == NS) { st = 0; par ^= 1; }
                if (HIST && (n + 1 == NQr || !mbar_test(&empty[st], par))) st_release_gpu(gp, n + 1);
            }
        }
        if ((DIR == 0 || meet) && a.beside_proj) {   // every tile of this side has been seen by lane 0: the same sum, `fr` is complete
            __syncwarp();
            double s = 0.0;
            for (int t = t_lo + lane; t < t_hi; t += 32) s += (double)__ldcg(&w.fr[(size_t)b * a.T + t].y);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                s += __hiloint2double(__shfl_xor_sync(FULL, __double2hiint(s), o), __shfl_xor_sync(FULL, __double2loint(s), o));
            }
            if (lane == 0) { sts_f64(lsum, s); sts_release(lsum + 8, 1); }
        }
        return;
    }

    // ---- walker warps ----
    const int* lab = FUSED ? slab : w.lab + (size_t)b * w.Lp;
    const int g0 = tid * P;
    const uint32_t bcol = (w.dense ? (uint32_t)a.blank : 0u) * (kEC * 8u);
    bool skip[P]; uint32_t ccol[P];
#pragma unroll
    for (int p = 0; p < P; ++p) {
        const int g = g0 + p;
        const bool vl = g < Lb;
        const int cur = vl ? (DIR ? lab[Lb - 1 - g] : lab[g]) : -1;
        const int prv = (vl && g >= 1) ? (DIR ? lab[Lb - g] : lab[g - 1]) : -2;
        skip[p] = vl && g >= 1 && cur != prv;
        ccol[p] = vl ? (w.dense ? (uint32_t)cur : (uint32_t)(DIR ? Lb - g : g + 1)) * (kEC * 8u) : bcol;
    }
    double bm[P], lm[P], fb[P], fls[P], flb[P]; int eb[P], el[P];
#pragma unroll
    for (int p = 0; p < P; ++p) {
        bm[p] = 0.0; lm[p] = 0.0; eb[p] = 0; el[p] = 0;
        fb[p] = 1.0; flb[p] = 1.0; fls[p] = skip[p] ? 1.0 : 0.0;
    }
    if (tid == 0) bm[0] = 1.0;                  // virtual alpha_{-1} = delta(s = 0)

    // history / offset rows of the current frame block: running pointers (dir 1 walks the blocks downwards)
    int2* hch = nullptr; int2* och = nullptr;
    constexpr long long kHistStep = (long long)kG * NW * PW, kOffStep = (long long)NW * PW;
    if (HIST) {
        const size_t blk0 = DIR ? (size_t)(NQ - 1) : 0;
        hch = (DIR ? w.hB : w.hA) + ((size_t)b * w.NB + blk0) * kG * NW * PW + g0;
        och = (DIR ? w.oB : w.oA) + ((size_t)b * w.NB + blk0) * NW * PW + g0;
    }

    const bool has_left = NW > 1 && warp > 0, has_right = NW > 1 && warp < NW - 1;
    const bool pub = has_right && lane == 31;
    const uint32_t my_halo = halo + warp * kHaloDepth * kG * 8;
    const uint32_t nb_halo = halo + (warp > 0 ? warp - 1 : 0) * kHaloDepth * kG * 8;
    const uint32_t my_meta = meta + warp * kHaloDepth * (uint32_t)sizeof(HaloMeta);
    const uint32_t nb_meta = meta + (warp > 0 ? warp - 1 : 0) * kHaloDepth * (uint32_t)sizeof(HaloMeta);
    const uint32_t nb_prog = prog + (warp > 0 ? warp - 1 : 0) * 4;
    double pm = 0.0;                            // left neighbour's label state for the coming step (lane 0: left warp's)
    int c_el = 0, c_R = 0, c_F = 0;             // left warp's meta as of my last renormalisation
    int Rout = 0, Fout = 0;                     // my scan carry / front offset for the right warp

    int st = 0, ph = 0;
    uint32_t stage_base = ring;
#pragma unroll 1
    for (int n = 0; n < NQr; ++n) {
        const int blk = DIR ? NQ - 1 - n : n;
        const int ns = blk == NQ - 1 ? rlast : kG;
        const uint32_t par = (uint32_t)(n & (kHaloDepth - 1));
        CTCB_TP(0);
        // the block is in shared memory long before it is needed (the ring runs many blocks ahead)
        mbar_wait(&full[st], ph);
        // emissions of the group's first step; every later step's are requested one step ahead
        const int j0 = DIR ? ns - 1 : 0;
        double yb, yl[P];
        yb = lds_f64(stage_base + bcol + (uint32_t)j0 * 8u);
#pragma unroll
        for (int p = 0; p < P; ++p) yl[p] = lds_f64(stage_base + ccol[p] + (uint32_t)j0 * 8u);
        // ---- between groups: everything that needs a branch ----
        // renormalise?  (some state drifted past 2^+-kDrift, or the left neighbour's offsets moved).
        // Positive doubles order like their high words; an exact zero (high word 0) never triggers.
        int bad = 0;
        {
            constexpr unsigned LO = (1023u - kDrift) << 20, SPAN = (2u * kDrift + 1u) << 20;
#pragma unroll
            for (int p = 0; p < P; ++p) {
                const unsigned hb = (unsigned)__double2hiint(bm[p]), hl = (unsigned)__double2hiint(lm[p]);
                bad |= (int)(hb != 0u) & (int)(hb - LO >= SPAN);
                bad |= (int)(hl != 0u) & (int)(hl - LO >= SPAN);
            }
        }
        if (has_left) { while (lds_acquire(nb_prog) < n + 1) { } }                    // left neighbour finished this group
        CTCB_TP(1);
        // left neighbour's state for this group (written at ITS group-n boundary)
        int m_el = 0, m_R = kZeroE, m_F = 0;
        if (has_left) {
            const uint32_t ma = nb_meta + par * (uint32_t)sizeof(HaloMeta);
            const double hal = lds_f64(ma);
            if (lane == 0) pm = hal;
            m_el = lds_relaxed(ma + 8); m_R = lds_relaxed(ma + 12); m_F = lds_relaxed(ma + 16);
            bad |= (m_el ^ c_el) | (m_R ^ c_R) | (m_F ^ c_F);
        }
        const bool trig = bad != 0;
        if (__builtin_expect(__any_sync(FULL, trig), 0)) {
            CTCB_TP(7);
            c_el = m_el; c_R = m_R; c_F = m_F;
            int natb[P], natl[P], am[P];
            bool hard = false;
#pragma unroll
            for (int p = 0; p < P; ++p) {
                natb[p] = bm[p] != 0.0 ? eb[p] + dexp(bm[p]) : kZeroE;
                natl[p] = lm[p] != 0.0 ? el[p] + dexp(lm[p]) : kZeroE;
                am[p] = max(natb[p], natl[p]);
                hard |= bm[p] == 0.0 || lm[p] == 0.0 || natb[p] - kD > natl[p];
            }
            {
                int pa = __shfl_up_sync(FULL, am[P - 1], 1);
                if (lane == 0) pa = m_R;
#pragma unroll
                for (int p = 0; p < P; ++p) { hard |= pa - kD > min(natb[p], natl[p]); pa = am[p]; }
            }
            if (__any_sync(FULL, hard)) {
                // R(g) = max(a(g), R(g-1) - kD): in the lane, then across lanes (decay P*kD per lane)
                int x = am[0], anymax = am[0];
#pragma unroll
                for (int p = 1; p < P; ++p) { x = max(am[p], x - kD); anymax = max(anymax, am[p]); }
#pragma unroll
                for (int i = 1; i < 32; i <<= 1) {
                    const int y = __shfl_up_sync(FULL, x, i);
                    if (lane >= i) x = max(x, y - i * P * kD);
                }
                x = max(max(x, m_R - (lane + 1) * P * kD), 2 * kZeroE);
                int Rp = __shfl_up_sync(FULL, x, 1);
                if (lane == 0) Rp = m_R;
                const unsigned nz = __ballot_sync(FULL, anymax > kZeroE);
                const int fl = nz ? 31 - __clz(nz) : -1;            // lane of the wavefront's last nonzero pair
                int F = m_F;
                if (nz) F = __shfl_sync(FULL, x, fl);
                Fout = F;
                Rout = (nz >> 31) ? __shfl_sync(FULL, x, 31) : kZeroE;
                const bool beyond = lane > fl;                      // exactly-zero states beyond the front take F
#pragma unroll
                for (int p = 0; p < P; ++p) {
                    const int base = Rp - kD;
                    const int zoff = beyond ? F : base;
                    const int neb = natb[p] > kZeroE ? max(natb[p], base) : zoff;
                    const int nel = natl[p] > kZeroE ? max(natl[p], max(natb[p] - kD, base)) : (natb[p] > kZeroE ? neb : zoff);
                    bm[p] *= pow2c(eb[p] - neb);
                    lm[p] *= pow2c(el[p] - nel);
                    eb[p] = neb; el[p] = nel;
                    Rp = max(max(am[p], Rp - kD), 2 * kZeroE);
                }
            } else {
                // plain drift: every exponent moves into its offset, no constraint is active
#pragma unroll
                for (int p = 0; p < P; ++p) {
                    bm[p] = dmant(bm[p]); lm[p] = dmant(lm[p]);
                    eb[p] = natb[p]; el[p] = natl[p];
                }
                Rout = __shfl_sync(FULL, am[P - 1], 31);
                Fout = Rout;
            }
            {                                                   // values moved: refresh the pre-shuffled neighbour
                const double q = shfl_up_f64(lm[P - 1]);
                if (lane != 0) pm = q;
            }
            int ep = __shfl_up_sync(FULL, el[P - 1], 1);
            if (lane == 0) ep = has_left ? m_el : eb[0];
#pragma unroll
            for (int p = 0; p < P; ++p) {
                fb[p] = pow2c(ep - eb[p]);
                fls[p] = skip[p] ? pow2c(ep - el[p]) : 0.0;
                flb[p] = pow2c(eb[p] - el[p]);
                ep = el[p];
            }
        }
        if (pub) {                                              // my state for the right neighbour's group n
            const uint32_t ma = my_meta + par * (uint32_t)sizeof(HaloMeta);
            sts_f64(ma, lm[P - 1]);
            sts_s32(ma + 8, el[P - 1]); sts_s32(ma + 12, Rout); sts_s32(ma + 16, Fout);
        }
        if (HIST) {
#pragma unroll
            for (int p = 0; p < P; ++p) och[p] = make_int2(eb[p], el[p]);
        }
        CTCB_TP(2);
        // halo slot of walking-order step s: dir 0 s = j, dir 1 s = ns-1-j
        const uint32_t hs_my = my_halo + par * (kG * 8u) + (DIR ? (uint32_t)(ns - 1) * 8u : 0u);
        const uint32_t hs_nb = nb_halo + par * (kG * 8u) + (DIR ? (uint32_t)(ns - 1) * 8u : 0u);
        // one recursion step on frame j of the block; so = halo slot offset of this step
        // The shuffle that feeds pair 0 is issued one step AHEAD, right after the lane's last pair
        // is updated: a warp issues in order, so a shuffle consumed in the step that issues it
        // would expose its full latency on every step.
        // A warp issues in order, so the source is written level by level (all pairs' first
        // FMAs, then the second, then the emission products): three dependent FP64 levels per step.
        // nj = frame of the NEXT step (its emissions are requested now), or -1 after the last one
        auto step = [&](int j, int nj, uint32_t so) {
            double hv = 0.0, nyb = 0.0, nyl[P];
            if (nj >= 0) {
                nyb = lds_f64(stage_base + bcol + (uint32_t)nj * 8u);
#pragma unroll
                for (int p = 0; p < P; ++p) nyl[p] = lds_f64(stage_base + ccol[p] + (uint32_t)nj * 8u);
            }
            if (has_left) hv = lds_f64(hs_nb + so);
            double t0[P], sb[P], sl[P];
#pragma unroll
            for (int p = P - 1; p >= 0; --p) {
                const double prev = p == 0 ? pm : lm[p - 1];
                t0[p] = fma(bm[p], flb[p], lm[p]);
                sb[p] = fma(prev, fb[p], bm[p]);
            }
#pragma unroll
            for (int p = P - 1; p >= 0; --p) {
                const double prev = p == 0 ? pm : lm[p - 1];
                sl[p] = fma(prev, fls[p], t0[p]);
            }
#pragma unroll
            for (int p = P - 1; p >= 0; --p) lm[p] = sl[p] * yl[p];
            const double pm_next = shfl_up_f64(lm[P - 1]);
            if (pub) sts_f64(hs_my + so, lm[P - 1]);
#pragma unroll
            for (int p = P - 1; p >= 0; --p) bm[p] = sb[p] * yb;
            if (HIST) {
                // history = the high words (exponent + 20 mantissa bits): the posteriors are ratios, the
                // truncation bias cancels and what is left is < 2^-20 relative (DESIGN.md section 4)
                int2 hw[P];
#pragma unroll
                for (int p = 0; p < P; ++p)
                    hw[p] = DIR ? make_int2(__double2hiint(sb[p]), __double2hiint(sl[p]))
                                : make_int2(__double2hiint(bm[p]), __double2hiint(lm[p]));
                int2* dst = hch + j * (NW * PW);
                if (P % 2 == 0) {
#pragma unroll
                    for (int p = 0; p < P; p += 2)
                        *reinterpret_cast<int4*>(dst + p) = make_int4(hw[p].x, hw[p].y, hw[(p + 1) % P].x, hw[(p + 1) % P].y);
                } else {
#pragma unroll
                    for (int p = 0; p < P; ++p) dst[p] = hw[p];
                }
            }
            pm = pm_next;
            if (lane == 0) pm = hv;
            if (nj >= 0) {
                yb = nyb;
#pragma unroll
                for (int p = 0; p < P; ++p) yl[p] = nyl[p];
            }
        };
        CTCB_TP(3);
        if (ns == kG) {
#pragma unroll
            for (int jj = 0; jj < kG; ++jj) {
                const int j = DIR ? kG - 1 - jj : jj;           // frame within the block
                const int nj = jj + 1 < kG ? (DIR ? j - 1 : j + 1) : -1;
                step(j, nj, DIR ? 0u - (uint32_t)j * 8u : (uint32_t)j * 8u);
            }
        } else {                                                // the utterance's partial block (once per walker)
#pragma unroll 1
            for (int jj = 0; jj < ns; ++jj) {
                const int j = DIR ? ns - 1 - jj : jj;
                const int nj = jj + 1 < ns ? (DIR ? j - 1 : j + 1) : -1;
                step(j, nj, DIR ? 0u - (uint32_t)j * 8u : (uint32_t)j * 8u);
            }
        }
        CTCB_TP(4);
        // publish: halo slots (and history), then the count; hand the ring stage back to the producer
        // (one warp barrier orders every lane's stage reads and history stores before both)
        __syncwarp();
        if (lane == 31) {
            if (NW > 1 || (FUSED && HIST)) sts_release(prog + warp * 4, n + 1);
            mbar_arrive(&empty[st]);
        }
        CTCB_TP(5);
        CTCB_TP(6);
        stage_base += stage_bytes;
        if (++st == NS) { st = 0; ph ^= 1; stage_base = ring; }
        if (HIST) { hch += DIR ? -kHistStep : kHistStep; och += DIR ? -kOffStep : kOffStep; }
    }

    if (meet) {
        // ---- hand over at the meeting frame m = 8 Mblk - 1: alpha_m (this walker's state) resp. beta'_m (the
        // reversed walker's sums BEFORE frame m's emission: one more transition-only step); mantissa + full exponent ----
        MeetSlot* mine = w.meet + ((size_t)b * 2 + DIR) * (NW * PW) + g0;
#pragma unroll
        for (int p = 0; p < P; ++p) {
            double vb = bm[p], vl = lm[p];
            if (DIR) {
                const double prev = p == 0 ? pm : lm[p - 1];
                const double t0 = fma(bm[p], flb[p], lm[p]);
                vb = fma(prev, fb[p], bm[p]);
                vl = fma(prev, fls[p], t0);
            }
            MeetSlot ms;
            ms.ob = vb != 0.0 ? eb[p] + dexp(vb) : kZeroE; ms.vb = vb != 0.0 ? dmant(vb) : 0.0;
            ms.ol = vl != 0.0 ? el[p] + dexp(vl) : kZeroE; ms.vl = vl != 0.0 ? dmant(vl) : 0.0;
            mine[p] = ms;
        }
        if (tid == 0) {                             // this side's sum of the frames' log2 normalisers
            double lz = 0.0;
            if (FUSED) {
#pragma unroll
                for (int q = 0; q < kFusedProducers * 8; ++q) lz += lds_f64(lsum + 16 + q * 8);
            } else {
                while (lds_acquire(lsum + 8) == 0) { }
                lz = lds_f64(lsum);
            }
            w.meetlz[2 * b + DIR] = lz;
        }
        __threadfence();
        __syncwarp();
        int old = 0;
        if (lane == 0) old = atomicAdd(w.meetcnt + b, 1);
        old = __shfl_sync(FULL, old, 0);
        if (old == 2 * NW - 1) {
            // the last warp of the utterance's two CTAs: P(l|x) = sum_g alpha_b(g) beta'_b(L-g) + sum_g alpha_l(g) beta'_l(L-1-g)
            // (the reversed walker's pair g holds the original lattice's blank L-g and label L-1-g)
            __threadfence();
            const MeetSlot* A = w.meet + (size_t)b * 2 * (NW * PW);
            const MeetSlot* Bq = A + NW * PW;
            int emax = 2 * kZeroE;
#pragma unroll 4                                    // four iterations' loads in flight: the slots come from L2
            for (int g = lane; g <= Lb; g += 32) {
                const int eA = __ldcg(&A[g].ob), eB = __ldcg(&Bq[Lb - g].ob);
                if (eA > kZeroE && eB > kZeroE) emax = max(emax, eA + eB);
                if (g < Lb) {
                    const int fA = __ldcg(&A[g].ol), fB = __ldcg(&Bq[Lb - 1 - g].ol);
                    if (fA > kZeroE && fB > kZeroE) emax = max(emax, fA + fB);
                }
            }
            emax = __reduce_max_sync(FULL, emax);
            double sum = 0.0;
#pragma unroll 4
            for (int g = lane; g <= Lb; g += 32) {
                const int eA = __ldcg(&A[g].ob), eB = __ldcg(&Bq[Lb - g].ob);
                if (eA > kZeroE && eB > kZeroE) sum += __ldcg(&A[g].vb) * __ldcg(&Bq[Lb - g].vb) * pow2c(eA + eB - emax);
                if (g < Lb) {
                    const int fA = __ldcg(&A[g].ol), fB = __ldcg(&Bq[Lb - 1 - g].ol);
                    if (fA > kZeroE && fB > kZeroE) sum += __ldcg(&A[g].vl) * __ldcg(&Bq[Lb - 1 - g].vl) * pow2c(fA + fB - emax);
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1)
                sum += __hiloint2double(__shfl_xor_sync(FULL, __double2hiint(sum), o), __shfl_xor_sync(FULL, __double2loint(sum), o));
            if (lane == 0) {
                const double lz = __ldcg(w.meetlz + 2 * b) + __ldcg(w.meetlz + 2 * b + 1);
                const double nll = -kLn2 * ((double)emax + log2(sum) - lz);
                a.loss[b] = (float)nll;
                if (a.loss_sum) atomicAdd(a.loss_sum, nll);
            }
        }
    } else if (DIR == 0) {
        // P(l|x) = alpha_{T-1}(2L) + alpha_{T-1}(2L-1) = the blank sum of slot L_b at a
        // virtual step T_b (pm already holds the neighbour's state after step T_b-1).
#pragma unroll
        for (int p = 0; p < P; ++p) {
            if (g0 + p == Lb) {
                const double prev = p == 0 ? pm : lm[p - 1];
                const double sb = fma(prev, fb[p], bm[p]);
                double lz = 0.0;
                if (FUSED) {
#pragma unroll
                    for (int q = 0; q < kFusedProducers * 8; ++q) lz += lds_f64(lsum + 16 + q * 8);
                } else {
                    while (lds_acquire(lsum + 8) == 0) { }
                    lz = lds_f64(lsum);
                }
                const double nll = -kLn2 * ((double)eb[p] + log2(sb) - lz);
                a.loss[b] = (float)nll;
                if (a.loss_sum) atomicAdd(a.loss_sum, nll);
            }
        }
    }
}

// DEC (fused, loss evaluation only): the producers also leave each valid frame's greedy-decode word (WalkArgs::dec)
template <int P, int NW, bool HIST, bool FUSED, typename LT = float, bool DEC = false>
__global__ void __launch_bounds__((NW + (FUSED ? kFusedProducers + 1 : 1)) * 32) k_walk(WalkArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    if (a.pdl_wait) asm volatile("griddepcontrol.wait;" ::: "memory");   // everything enqueued before this kernel is complete and visible
    const int b = blockIdx.x;
    if (!FUSED) {
        // the gradient kernel may start as soon as every walker CTA is resident: its CTAs wait per
        // frame block on the progress this kernel publishes (Workspace::gprog)
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        if (a.beside_proj) {                    // the metadata kernel ran before the projection: its word is set, with release
            if (threadIdx.x == 0) {
                const long long t0 = clock64();
                while (ld_acquire_gpu(a.w.gprog + 4 * b + 2) != a.w.stamp && clock64() - t0 < kSpinLimit) __nanosleep(256);
            }
            __syncthreads();
        }
        const int flags = __ldcg(a.w.flags + b), Tb = __ldcg(a.w.Tb + b), Lb = __ldcg(a.w.Lb + b);
        if (flags & UTT_INFEASIBLE) return;
        if (blockIdx.y == 0) walk_dir<P, NW, 0, HIST, false>(a, smem_raw, Tb, Lb, flags);
        else                 walk_dir<P, NW, 1, HIST, false>(a, smem_raw, Tb, Lb, flags);
        return;
    }
    // ---- fused variant: no k_emit ran.  Rows a3/a5 (operator parameter layer, lattice metadata)
    // are derived here by every walker CTA for itself. ----
    const Problem& p = a.p;
    const Workspace& w = a.w;
    const int tid = threadIdx.x, nthr = blockDim.x;
    __shared__ int s_L, s_rep, s_flags;
    if (tid == 0) {
        // the progress words of this call start at 0 BEFORE any gradient CTA can exist
        w.gprog[4 * b + blockIdx.y] = 0;
        if (blockIdx.y == 0) { w.gprog[4 * b + 2] = 0; w.gprog[4 * b + 3] = 0; }
        __threadfence();
        s_L = p.Lmax; s_rep = 0; s_flags = 0;
    }
    __syncthreads();
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    int Tb = p.T, lenflags = 0;
    if (p.data_len) {
        long long t64 = load_as_int(p.data_len, p.data_len_dtype, b);
        if (t64 < 0) { t64 = 0; lenflags = UTT_LEN_CLAMPED; }
        if (t64 > p.T) { t64 = p.T; lenflags = UTT_LEN_CLAMPED; }
        Tb = (int)t64;
    }
    int L;
    if (p.label_len) {
        long long l64 = load_as_int(p.label_len, p.label_len_dtype, b);
        if (l64 < 0) { l64 = 0; lenflags = UTT_LEN_CLAMPED; }
        if (l64 > p.Lmax) { l64 = p.Lmax; lenflags = UTT_LEN_CLAMPED; }
        L = (int)l64;
    } else {
        for (int j = tid; j < p.Lmax; j += nthr)
            if (load_as_int(p.labels, p.label_dtype, b * p.lst_b + j * p.lst_l) == p.label_pad) atomicMin(&s_L, j);
        __syncthreads();
        L = s_L;
    }
    // the labels live behind the walker's other shared-memory regions (same carve as walk_dir)
    int* slab;
    {
        const size_t stage_bytes = (size_t)w.W * kEC * 8;
        size_t off = (size_t)a.stages * stage_bytes + 2 * kMaxStages * sizeof(uint64_t) +
                     (size_t)NW * kHaloDepth * kG * 8 + (size_t)NW * kHaloDepth * sizeof(HaloMeta) + (size_t)NW * 4;
        off = (off + 7) & ~(size_t)7;
        slab = reinterpret_cast<int*>(smem_raw + off + 32 + kFusedProducers * 64);
    }
    {
        int bad = 0;
        for (int j = tid; j < L; j += nthr) {
            long long v = load_as_int(p.labels, p.label_dtype, b * p.lst_b + j * p.lst_l);
            if (v < 0 || v >= p.V || v == p.blank) bad = 1;
            slab[j] = (int)(v < 0 ? 0 : (v >= p.V ? p.V - 1 : v));
        }
        if (bad) atomicOr(&s_flags, UTT_BAD_LABEL);
    }
    __syncthreads();
    {
        int rep = 0;
        for (int j = tid + 1; j < L; j += nthr) rep += slab[j] == slab[j - 1];
        if (rep) atomicAdd(&s_rep, rep);
    }
    __syncthreads();
    int flags = s_flags | lenflags;
    if (Tb <= 0 || L + s_rep > Tb) flags |= UTT_INFEASIBLE;
    if (blockIdx.y == 0 && tid == 0) {
        if (p.status) p.status[b] = flags;
        if (flags & UTT_INFEASIBLE) {
            p.loss[b] = 0.0f;                        // defined behaviour, SURVEY 7.3-6
            w.Tb[b] = Tb; w.Lb[b] = L; w.flags[b] = flags; w.nd[b] = 0;
            st_release_gpu(w.gprog + 4 * b + 2, w.stamp);
        } else if (!HIST) {
            w.Tb[b] = Tb; w.Lb[b] = L; w.flags[b] = flags;
        }
    }
    if (flags & UTT_INFEASIBLE) {
        // no producers run, but hypotheses do not depend on the labels: the alpha CTA decodes the frames, a warp per frame
        if (DEC && blockIdx.y == 0)
            greedy_frames(utt_logits<LT>(p, b), 0, p.st_t, Tb, p.V, tid >> 5, nthr >> 5, tid & 31,
                          [&](int t, const Top2& tp) { a.dec.tok[(size_t)b * p.T + t] = decode_word(tp, a.dec.unk); });
        return;
    }
    if (blockIdx.y == 0) walk_dir<P, NW, 0, HIST, true, LT, DEC>(a, smem_raw, Tb, L, flags);
    else                 walk_dir<P, NW, 1, HIST, true, LT, DEC>(a, smem_raw, Tb, L, flags);
}

// the walker configurations {P, NW} the library instantiates (ctcb.cu's table, ctcb_decode.cu's decoding variants)
#define CTCB_WALK_CONFIGS(X) X(1, 1) X(2, 1) X(4, 1) X(1, 2) X(2, 2) X(4, 2) X(1, 3) X(2, 3) X(4, 3) \
    X(1, 4) X(2, 4) X(4, 4) X(2, 5) X(2, 6) X(1, 8) X(2, 8) X(4, 8) X(2, 12) X(2, 16) X(4, 16)

// host side: the decoding instantiations (k_walk<P, NW, false, true, LT, true> and k_emit<VEC, NQ, LT, true>) are compiled
// in a translation unit of their own, ctcb_decode.cu, which hands their addresses to ctcb.cu's launch path
using WalkKernel = void (*)(WalkArgs);
using EmitKernel = void (*)(Problem, Workspace, DecodeOut);
WalkKernel walk_decode_kernel(int P, int NW, bool bf16);    // nullptr for a configuration outside CTCB_WALK_CONFIGS
EmitKernel emit_decode_kernel(int vec, int nq, bool bf16);  // nq: -1 staged (vec 4), 0 two-pass, 1..16 register-resident

// ---------------------------------------------------------------------------------------
// k_mailbox_exchange: the loss-sum exchange of section 8e over NVLink peer memory.  One warp.
// Exchange k of a rank (k = its device-side counter): lane r takes rank r's row of exchange k-lag
// from the LOCAL mailbox (acquire; the peers stored it `lag` exchanges ago, so the wait is normally
// over before it starts) and lane 0 adds the rows in rank order -- every rank forms the same sum
// with the same bits; lane r then stores this rank's partial sums into rank r's mailbox (slot
// k mod 2*lag, row = this rank) with a release at system scope.  No NCCL kernel, no rendezvous on
// the step's path: `lag` steps of slack between the ranks, for loops whose step times differ from
// rank to rank and step to step (bench.py's uniform shards measure the same with lag 1, 4 and 8;
// DESIGN.md section 8).  A peer that never shows up ends the wait
// after ~2 s with NaN instead of hanging the GPU.
// ---------------------------------------------------------------------------------------
constexpr int kMailMaxRanks = 16, kMailMaxCount = 6, kMailRow = 8;      // row: 6 values, pad, sequence number
constexpr int kMailMaxLag = 8;
struct MailboxDev {
    double* peer[kMailMaxRanks];        // rank r's mailbox as mapped into this process ([2*lag][world][kMailRow] doubles)
    unsigned long long* counter;        // exchanges done by this rank
    int rank, world;
    int lag;                            // exchange k returns the sums of exchange k - lag: the ranks' slack, in steps
};

// what the kernel's one warp does
__device__ __forceinline__ void mailbox_exchange_warp(const MailboxDev* md, double* values, int count, double* out, int flush, int lane) {
    const MailboxDev& m = *md;
    const unsigned long long k = *m.counter;          // exchanges completed so far = index of this one
    __shared__ double rows[kMailMaxRanks][kMailMaxCount];
    __shared__ int timed_out;
    // a wait that timed out once poisons the mailbox: later exchanges report NaN at once instead of waiting again
    if (lane == 0) timed_out = m.counter[1] != 0ull;
    __syncwarp();
    // 1. gather exchange k-lag (flush: the last one, k-1) from the local mailbox.  Gather BEFORE publish: a peer
    //    that stores exchange j has gathered this rank's exchange j-lag, so j <= k-1+lag while this rank is still
    //    reading slot (k-lag) mod S -- with S = 2*lag slots the peer's store cannot land on that slot.
    const unsigned long long back = flush ? 1ull : (unsigned long long)m.lag;
    const unsigned S = 2u * (unsigned)m.lag;
    const bool have = k >= back;
    if (have && lane < m.world) {
        const unsigned long long kk = k - back;
        const double* src = m.peer[m.rank] + ((size_t)(kk % S) * m.world + lane) * kMailRow;
        const unsigned long long* seq = reinterpret_cast<const unsigned long long*>(src + kMailRow - 1);
        const long long t0 = clock64();
        for (; !timed_out;) {
            unsigned long long got;
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(got) : "l"(seq) : "memory");
            if (got >= kk + 1) break;
            if (clock64() - t0 > 4000000000LL) { timed_out = 1; break; }
            __nanosleep(200);
        }
        for (int c = 0; c < count; ++c) {
            double v; asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(src + c) : "memory");
            rows[lane][c] = v;
        }
    }
    __syncwarp();
    if (lane == 0) {
        for (int c = 0; c < count; ++c) {
            double s = 0.0;
            if (have) for (int r = 0; r < m.world; ++r) s += rows[r][c];            // rank order: same bits on every rank
            out[c] = timed_out ? __longlong_as_double(0x7ff8000000000000LL) : s;
        }
        if (timed_out) m.counter[1] = 1ull;
    }
    if (flush) return;                                 // flush: read the last exchange only
    // 2. publish this rank's partial sums of exchange k into every rank's mailbox (its own included)
    if (lane < m.world) {
        double* dst = m.peer[lane] + ((size_t)(k % S) * m.world + m.rank) * kMailRow;
        for (int c = 0; c < count; ++c) asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(dst + c), "d"(values[c]) : "memory");
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(reinterpret_cast<unsigned long long*>(dst + kMailRow - 1)), "l"(k + 1) : "memory");
    }
    __syncwarp();
    if (lane == 0) {
        for (int c = 0; c < count; ++c) values[c] = 0.0;
        *m.counter = k + 1;
    }
}

#ifndef CTCB_NO_PLAIN_KERNELS   // non-template kernels: defined in ctcb.cu's translation unit only
__global__ void __launch_bounds__(32) k_mailbox_exchange(const MailboxDev* m, double* values, int count, double* out, int flush) {
    // Riding on a step, either BEHIND its gradient kernel as that kernel's programmatic dependent (this grid starts when
    // the gradient kernel's last wave of CTAs has started, works beside it -- it shares nothing with the step -- and stays
    // open until the step is complete and flushed, so the stream's next kernel sees both), or AHEAD of a forward-only
    // call, whose recursion kernel is then this grid's programmatic dependent and starts at once.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    mailbox_exchange_warp(m, values, count, out, flush, threadIdx.x);
    if (threadIdx.x == 0) asm volatile("griddepcontrol.wait;" ::: "memory");
}
#endif

// ---------------------------------------------------------------------------------------
// k_grad<VEC,CH,XQ>: grid (NB, B), block 128: one frame block (kG = 8 frames) per CTA, two
// frames per warp.  Rows a7 (accumulation, gradient) and a8 (head-gradient scaling), written
// once in the caller's layout.
// CH = register-resident chunks of 32 state pairs per lane (pairs <= 32*CH); CH = 0 is the
// generic two-pass variant for longer label sequences.  With CH <= 4 both frames of a warp are
// in flight together (every global load of the two frames is issued before the first use).
//
// State weights come from the walkers' high-word history: mantissa (20 bits) -> float in
// [1,2) by integer ops, exponent field + the frame block's offsets -> one integer per state;
// gamma_t(s) = alpha_t(s) beta'_t(s) / Z_t is normalised per frame from those integers, so
// nothing large is ever subtracted.  The offsets of alpha and beta' are combined once per
// warp (they are constant over the frame block).
// ---------------------------------------------------------------------------------------
struct GradArgs { Problem p; Workspace w; };

template <int VEC, typename LT>
__device__ __forceinline__ void zero_row(LT* row, int V, int lane) {
    using V_t = typename LV<LT, VEC>::type;
    const int nvec = V / VEC;
    V_t z; memset(&z, 0, sizeof(z));
    V_t* rv = reinterpret_cast<V_t*>(row);
    for (int k = lane; k < nvec; k += 32) rv[k] = z;
    for (int v = nvec * VEC + lane; v < V; v += 32) stx(row + v, 0.0f);
}

constexpr int kNoState = INT_MIN / 2;

// high word of a positive fp64 -> its 20 mantissa bits as a float in [1,2)
__device__ __forceinline__ float hw_mant(int h) { return __int_as_float(((h & 0x000fffff) << 3) | 0x3f800000); }
// alpha's high word after an exponent shift was added to it (k_grad2, k_meet, k_proj_occ): kept while it is a normal positive
// double, else 0 -- below the normal range (an occupancy below 2^-1022 times the largest beta'; a negative word when the
// shift wrapped) and at exponent 2047 (inf / NaN).  The latter is reached only by a state whose beta' is exactly 0 (every
// other state's occupancy is <= 1), where inf * 0 would be NaN; the product is 0 there
__device__ __forceinline__ int hw_normal_or_zero(int h) { return (unsigned)h - (1u << 20) < 0x7FE00000u ? h : 0; }
// weight (mantissa product in [1,4), total exponent) of alpha*beta' for one state; an exactly-zero
// factor (high word 0) gives the exponent kNoState, which xscale0 turns into weight 0
__device__ __forceinline__ void hw_weight(int ha, int hb, int off, float& wgt, int& e) {
    wgt = hw_mant(ha) * hw_mant(hb);
    e = min((unsigned)ha, (unsigned)hb) == 0u ? kNoState : (ha >> 20) + (hb >> 20) + off;
}

constexpr int kGradFramesPerWarp = 2;  // 4 warps x 2 frames = one frame block per CTA

// occupancy row of one frame in rank order: Lp label slots, or a slot per register-resident pair
__host__ __device__ inline int grad_row_floats(int Lp, int pairs_cap) { return ((Lp > pairs_cap ? Lp : pairs_cap) + 3) & ~3; }
// staged_V != 0: the frame block's kG logits rows are staged in shared memory (XQ < 0)
__host__ __device__ inline size_t grad_staged_bytes(int staged_V) { return staged_V ? (size_t)kG * staged_V * 4 + 64 : 0; }
__host__ __device__ inline size_t grad_smem_bytes(int Lp, int pairs_cap, int staged_V = 0) {
    return grad_staged_bytes(staged_V) + (size_t)(Lp + 1) * 8 + (size_t)4 * kGradFramesPerWarp * grad_row_floats(Lp, pairs_cap) * 4 + 16;
}

// XQ = VEC-wide loads per lane that hold the frame's logits row in registers (issued together
// with the history loads so that one memory round trip covers both); 0 = row loaded when needed;
// -1 (wide vocabularies, 16-byte aligned rows): the CTA's kG rows are fetched into shared memory by
// 1-D bulk copies (TMA) issued before anything else -- 8 rows in flight per CTA, several CTAs per SM,
// while the occupancies are computed -- the gradient row is formed in place, label columns included,
// and leaves with one bulk store per row.
// OCC = 1: registers capped at 64 (8 CTAs per SM instead of 7, a few spilled words) for batches
// that run after the walkers: measured -14 % at cfg5, but +5 % on the overlapped cfg2 step, where
// the kernel shares the GPU with the walkers and its tail is what counts -- hence a variant.
template <int VEC, int CH, int XQ, int OCC = 0, typename LT = float>
__global__ void __launch_bounds__(XQ < 0 ? 256 : 128, XQ < 0 ? (CH == 16 ? 2 : 3) : ((CH == 0 || CH == 8) ? 5 : (CH <= 4 ? (OCC ? 8 : 1) : 3))) k_grad(GradArgs a) {
    using V_t = typename LV<LT, VEC>::type;
    constexpr int NCH = CH > 0 ? CH : 1, NXQ = XQ > 0 ? XQ : 1;
    // staged rows: 8 warps, one frame each (the compute phase is latency-bound: twice the warps per SM)
    constexpr int FPW = XQ < 0 ? 1 : kGradFramesPerWarp, NT = XQ < 0 ? 256 : 128;
    constexpr int F = (CH > 0 && CH <= 4) ? FPW : 1;      // frames in flight per warp
    const Problem& p = a.p; const Workspace& w = a.w;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // a loss-sum exchange launched behind this grid as its programmatic dependent may start once every CTA is here
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // the utterance's metadata is written by k_emit (complete before this grid exists) or, in the
    // fused path, by the concurrently running alpha walker CTA
    // Both waits are bounded: a workspace that no matching forward call filled (another shape, other layout
    // switches, a forward that failed) makes this CTA write NaN into its rows and leave instead of hanging the GPU.
    __shared__ int s_ok;
    constexpr bool STAGED = XQ < 0;
    // Staged rows are the wide-vocabulary path: never the fused one, so everything k_emit wrote is complete before this grid
    // exists.  The stamp, the lengths, the flags, the distinct-label table and the rank order are then requested together --
    // one memory round trip instead of four dependent ones (the kernel's CTAs are short, under load a round trip is microseconds)
    int Tb_e = 0, Lb_e = 0, fl_e = 0, nd_e = 0, rk_e[NCH];
    extern __shared__ __align__(128) unsigned char gsm_all[];
    if (STAGED) {
        const int st = __ldcg(w.gprog + 4 * b + 2);
        Tb_e = __ldcg(w.Tb + b); Lb_e = __ldcg(w.Lb + b); fl_e = __ldcg(w.flags + b); nd_e = __ldcg(w.nd + b);
        const int* rank_e = w.rank + (size_t)b * w.Lp;
#pragma unroll
        for (int c = 0; c < NCH; ++c) rk_e[c] = __ldcg(rank_e + min(c * 32 + lane, w.Lp - 1));
        int2* s_dl_e = reinterpret_cast<int2*>(reinterpret_cast<float*>(gsm_all + grad_staged_bytes(p.V)) +
                                               (size_t)4 * kGradFramesPerWarp * grad_row_floats(w.Lp, 32 * CH));
        const int2* dl = w.dl + (size_t)b * (w.Lp + 1);
        for (int j = tid; j <= w.Lp; j += NT) s_dl_e[j] = __ldcg(dl + j);
        if (tid == 0) s_ok = st == w.stamp;
    } else if (tid == 0) {
        const long long t0 = clock64();
        int v;
        while ((v = ld_acquire_gpu(w.gprog + 4 * b + 2)) == 0 && clock64() - t0 < kSpinLimit) __nanosleep(256);
        s_ok = v == w.stamp;
    }
    __syncthreads();
    if (!s_ok) {
        for (int j = warp; j < kG; j += (XQ < 0 ? 8 : 4)) {
            const int t = blockIdx.y * kG + j;
            if (t < p.T) {
                LT* grow = grad_row<LT>(p, b, t);
                for (int v = lane; v < p.V; v += 32) stx(grow + v, __int_as_float(0x7fc00000));
            }
        }
        return;
    }
    const int Tb = STAGED ? Tb_e : __ldcg(w.Tb + b), Lb = STAGED ? Lb_e : __ldcg(w.Lb + b);
    const bool infeasible = ((STAGED ? fl_e : __ldcg(w.flags + b)) & UTT_INFEASIBLE) != 0;
    // CTAs are dispatched utterance-fastest, and per utterance in the order the walkers complete
    // the frame blocks: the two walkers meet in the middle, so from the middle outwards
    const int NQ = infeasible ? 0 : (Tb + kG - 1) / kG;
    int blk = blockIdx.y;
    if (blk < NQ) blk = (blk & 1) ? NQ / 2 - (blk + 1) / 2 : NQ / 2 + blk / 2;
    const float head = p.head ? p.head[b] : 1.0f;
    const int t_first = blk * kG;
    const bool cta_live = blk < NQ;
    const int GW = grad_row_floats(w.Lp, 32 * CH);
    unsigned char* gsm_raw = gsm_all + (STAGED ? grad_staged_bytes(p.V) : 0);
    float* srow = reinterpret_cast<float*>(gsm_all);                                         // kG rows of V floats
    uint64_t* rbar = reinterpret_cast<uint64_t*>(gsm_all + (size_t)kG * p.V * 4);            // one barrier per row
    if (STAGED && cta_live && lane == 0) {
        // this warp's rows: requested now, consumed after the occupancies of their frames
#pragma unroll
        for (int f = 0; f < FPW; ++f) mbar_init(rbar + warp * FPW + f, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#pragma unroll
        for (int f = 0; f < FPW; ++f) {
            const int j = warp * FPW + f, t = t_first + j;
            if (t < Tb) {
                // a bf16 row lands in the upper half of its fp32 slot and is widened in place (below)
                mbar_expect_tx(rbar + j, (uint32_t)p.V * (uint32_t)sizeof(LT));
                tma_load_1d(reinterpret_cast<LT*>(srow + (size_t)j * p.V) + (sizeof(LT) == 4 ? 0 : p.V),
                            utt_logits<LT>(p, b) + (long long)t * p.st_t, (uint32_t)p.V * (uint32_t)sizeof(LT), rbar + j);
            }
        }
    }
    float* gbuf0 = reinterpret_cast<float*>(gsm_raw) + (size_t)warp * FPW * GW;
    int2* s_dl = reinterpret_cast<int2*>(reinterpret_cast<float*>(gsm_raw) + (size_t)4 * kGradFramesPerWarp * GW);   // Lp + 1
    const int* rank = w.rank + (size_t)b * w.Lp;
    int nd = 0;
    if (cta_live) {
        if (STAGED) nd = nd_e;
        else {
            nd = __ldcg(w.nd + b);
            const int2* dl = w.dl + (size_t)b * (w.Lp + 1);
            for (int j = tid; j <= nd; j += NT) s_dl[j] = __ldcg(dl + j);
        }
        // block n is frame block n of the alpha walker and block NQ-1-n of the beta walker
        const int* gp = w.gprog + 4 * b;
        if (tid == 0) {
            const long long t0 = clock64();
            // back-off between polls: the pollers' traffic is not free for the walkers (profiles/r4r_poll_sweep.log: on the
            // wide-vocabulary path, whose gradient CTAs share the walkers' SMs, 64 ns costs 11 us per cfg3 step, 1024 ns saves 3)
            const unsigned pns = w.poll_ns > 0 ? (unsigned)w.poll_ns : (STAGED ? 1024u : 256u);
            while (ld_acquire_gpu(gp) < blk + 1 && clock64() - t0 < kSpinLimit) __nanosleep(pns);
            while (ld_acquire_gpu(gp + 1) < NQ - blk && clock64() - t0 < kSpinLimit) __nanosleep(pns);
            if (clock64() - t0 >= kSpinLimit) s_ok = 0;
        }
    }
    __syncthreads();
    if (!s_ok) {                                   // the recursion kernel never got there: NaN rows, no hang
        if (STAGED && lane == 0) {
#pragma unroll
            for (int f = 0; f < FPW; ++f) if (t_first + warp * FPW + f < Tb) mbar_wait(rbar + warp * FPW + f, 0);   // rows in flight land first
        }
        for (int j = warp; j < kG; j += NT / 32) {
            const int t = t_first + j;
            if (t < p.T) {
                LT* grow = grad_row<LT>(p, b, t);
                for (int v = lane; v < p.V; v += 32) stx(grow + v, __int_as_float(0x7fc00000));
            }
        }
        return;
    }

    const int pairs = 32 * w.P * w.NW;
    const size_t blkoff = (size_t)b * w.NB + blk;
    const int2* hA0 = w.hA + blkoff * kG * pairs;
    const int2* hB0 = w.hB + blkoff * kG * pairs;
    const int2* oA = w.oA + blkoff * pairs;
    const int2* oB = w.oB + blkoff * pairs;
    // alpha pair g <-> beta' pairs: blank of pair g = reversed-walker blank of slot L-g, label of
    // pair g = reversed-walker label of slot L-1-g.  Per lane and chunk, once per frame block: the
    // (clamped) history indices, the combined offsets -- kNoState for pairs beyond the lattice,
    // whose history is never masked by the walkers -- and the slot of the label state in rank order.
    int ibb[NCH], ibl[NCH], ofb[NCH], ofl[NCH], rk[NCH];
    int2 pha[NCH]; int phbb[NCH], phbl[NCH];
    if (STAGED && CH > 0 && cta_live) {
        // staged rows, one frame per warp: the warp's history loads go first, then the block's offsets -- ONCE per CTA, through
        // shared memory (the occupancy rows' space, not yet in use), instead of three gathers per chunk in each of the 8 warps
        // whose arrival the history loads had to wait for
        const int tq = t_first + warp;
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            const int g = c * 32 + lane;
            ibb[c] = max(Lb - g, 0); ibl[c] = max(Lb - 1 - g, 0);
            pha[c] = make_int2(0, 0); phbb[c] = 0; phbl[c] = 0;
        }
        if (tq < Tb) {
            const int2* A = hA0 + (size_t)(tq - t_first) * pairs + lane;
            const int2* Bh = hB0 + (size_t)(tq - t_first) * pairs;
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
                pha[c] = __ldcg(A + c * 32);
                phbb[c] = __ldcg(&Bh[ibb[c]].x);
                phbl[c] = __ldcg(&Bh[ibl[c]].y);
            }
        }
        int2* s_off = reinterpret_cast<int2*>(gsm_raw);          // [0, 32 CH): alpha walker's offsets, [32 CH, 64 CH): beta walker's
        for (int g = tid; g < 32 * NCH; g += NT) {
            s_off[g] = g < pairs ? __ldcg(oA + g) : make_int2(0, 0);
            s_off[32 * NCH + g] = g < pairs ? __ldcg(oB + g) : make_int2(0, 0);
        }
        __syncthreads();
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            const int g = c * 32 + lane;
            const int2 oa = s_off[g];
            const int ob = s_off[32 * NCH + ibb[c]].x, ol = s_off[32 * NCH + ibl[c]].y;
            ofb[c] = g <= Lb ? oa.x + ob : kNoState;
            ofl[c] = g < Lb ? oa.y + ol : kNoState;
            rk[c] = g < Lb ? rk_e[c] : g;
        }
        __syncthreads();                                          // the occupancy rows may be written from here on
    } else if (CH > 0 && cta_live) {
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            const int g = c * 32 + lane;
            ibb[c] = max(Lb - g, 0); ibl[c] = max(Lb - 1 - g, 0);
            const int2 oa = __ldcg(oA + g);
            const int ob = __ldcg(&oB[ibb[c]].x), ol = __ldcg(&oB[ibl[c]].y);
            ofb[c] = g <= Lb ? oa.x + ob : kNoState;
            ofl[c] = g < Lb ? oa.y + ol : kNoState;
            rk[c] = g < Lb ? (STAGED ? rk_e[c] : __ldcg(rank + g)) : g;
        }
    }
    const int nvec = p.V / VEC;

#pragma unroll
    for (int r = 0; r < FPW / F; ++r) {
        int tt[F]; bool live[F];
        int2 ha[F][NCH]; int hbb[F][NCH], hbl[F][NCH];
        V_t xr[F][NXQ]; float2 fr[F];
        // ---- every global load of the F frames ----
#pragma unroll
        for (int f = 0; f < F; ++f) {
            tt[f] = t_first + warp * FPW + r * F + f;
            live[f] = cta_live && tt[f] < Tb;
            fr[f] = make_float2(0.0f, 0.0f);
            if (live[f]) {
                fr[f] = __ldcg(w.fr + (size_t)b * p.T + tt[f]);
                const LT* xrow = utt_logits<LT>(p, b) + (long long)tt[f] * p.st_t;
                if (XQ > 0) {
                    const V_t* xv = reinterpret_cast<const V_t*>(xrow);
#pragma unroll
                    for (int q = 0; q < NXQ; ++q) { const int k = q * 32 + lane; xr[f][q] = k < nvec ? __ldg(xv + k) : LV<LT, VEC>::fill(0.0f); }
                }
                if (CH > 0) {
                    const int2* A = hA0 + (size_t)(tt[f] - t_first) * pairs + lane;
                    const int2* Bh = hB0 + (size_t)(tt[f] - t_first) * pairs;
#pragma unroll
                    for (int c = 0; c < NCH; ++c) {
                        if (STAGED) { ha[f][c] = pha[c]; hbb[f][c] = phbb[c]; hbl[f][c] = phbl[c]; continue; }
                        ha[f][c] = __ldcg(A + c * 32);
                        hbb[f][c] = __ldcg(&Bh[ibb[c]].x);
                        hbl[f][c] = __ldcg(&Bh[ibl[c]].y);
                    }
                }
            }
        }
        // ---- per frame: occupancy, softmax, gradient row ----
#pragma unroll
        for (int f = 0; f < F; ++f) {
            const int t = tt[f];
            if (t >= p.T) continue;
            LT* grow = grad_row<LT>(p, b, t);
            if (!live[f]) { zero_row<VEC>(grow, p.V, lane); continue; }
            const LT* xrow = utt_logits<LT>(p, b) + (long long)t * p.st_t;
            float* gbuf = gbuf0 + (size_t)(r * F + f) * GW;
            float zb = 0.0f, zl = 0.0f;
            if (CH > 0) {
                float wb[NCH], wl[NCH]; int eb[NCH], el[NCH];
                int emax = INT_MIN;
#pragma unroll
                for (int c = 0; c < NCH; ++c) {
                    hw_weight(ha[f][c].x, hbb[f][c], ofb[c], wb[c], eb[c]);
                    hw_weight(ha[f][c].y, hbl[f][c], ofl[c], wl[c], el[c]);
                    emax = max(emax, max(eb[c], el[c]));
                }
                emax = __reduce_max_sync(0xffffffffu, emax);
#pragma unroll
                for (int c = 0; c < NCH; ++c) {
                    zb += xscale0(wb[c], eb[c] - emax);
                    const float v = xscale0(wl[c], el[c] - emax);
                    zl += v;
                    gbuf[rk[c]] = v;
                }
            } else {
                const int2* A = hA0 + (size_t)(t - t_first) * pairs;
                const int2* Bh = hB0 + (size_t)(t - t_first) * pairs;
                int emax = INT_MIN;
                for (int g = lane; g <= Lb; g += 32) {
                    const int2 av = __ldcg(A + g), oa = __ldcg(oA + g);
                    float wgt; int e;
                    hw_weight(av.x, __ldcg(&Bh[Lb - g].x), oa.x + __ldcg(&oB[Lb - g].x), wgt, e);
                    emax = max(emax, e);
                    if (g < Lb) { hw_weight(av.y, __ldcg(&Bh[Lb - 1 - g].y), oa.y + __ldcg(&oB[Lb - 1 - g].y), wgt, e); emax = max(emax, e); }
                }
                emax = __reduce_max_sync(0xffffffffu, emax);
                for (int g = lane; g <= Lb; g += 32) {
                    const int2 av = __ldcg(A + g), oa = __ldcg(oA + g);
                    float wgt; int e;
                    hw_weight(av.x, __ldcg(&Bh[Lb - g].x), oa.x + __ldcg(&oB[Lb - g].x), wgt, e);
                    zb += xscale0(wgt, e - emax);
                    if (g < Lb) {
                        hw_weight(av.y, __ldcg(&Bh[Lb - 1 - g].y), oa.y + __ldcg(&oB[Lb - 1 - g].y), wgt, e);
                        const float v = xscale0(wgt, e - emax);
                        zl += v; gbuf[__ldcg(rank + g)] = v;
                    }
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                zb += __shfl_xor_sync(0xffffffffu, zb, o);
                zl += __shfl_xor_sync(0xffffffffu, zl, o);
            }
            const float rZ = 1.0f / (zb + zl);
            const float gblank = zb * rZ;
            __syncwarp();
            // dense row: head * softmax, blank column corrected
            const float fmx = fr[f].x, flz = fr[f].y;
            V_t* gv = reinterpret_cast<V_t*>(grow);
            if (XQ > 0) {
#pragma unroll
                for (int q = 0; q < NXQ; ++q) {
                    const int k = q * 32 + lane;
                    if (k < nvec) {
                        float x[VEC]; LV<LT, VEC>::get(xr[f][q], x);
                        float y[VEC];
#pragma unroll
                        for (int j = 0; j < VEC; ++j) {
                            y[j] = fast_ex2(fmaf(x[j] - fmx, kLog2e, -flz));
                            if (k * VEC + j == p.blank) y[j] -= gblank;
                            y[j] *= head;
                        }
                        gv[k] = LV<LT, VEC>::pack(y);
                    }
                }
            } else if (STAGED) {
                // the row is in shared memory: gradient formed in place, then one bulk store
                float* sr = srow + (size_t)(warp * FPW + r * F + f) * p.V;
                mbar_wait(rbar + warp * FPW + r * F + f, 0);
                float4* sv = reinterpret_cast<float4*>(sr);
                if constexpr (sizeof(LT) == 4) {
                    for (int k = lane; k < nvec; k += 32) {
                        float4 v = sv[k];
                        v.x = head * fast_ex2(fmaf(v.x - fmx, kLog2e, -flz));
                        v.y = head * fast_ex2(fmaf(v.y - fmx, kLog2e, -flz));
                        v.z = head * fast_ex2(fmaf(v.z - fmx, kLog2e, -flz));
                        v.w = head * fast_ex2(fmaf(v.w - fmx, kLog2e, -flz));
                        sv[k] = v;
                    }
                } else {
                    // bf16 row in the upper half of the slot, widened in place to the fp32 row head * y: the fp32 elements
                    // 4k..4k+3 overwrite bf16 elements <= 4k+3 only, which this step (all loads before the warp's stores)
                    // or an earlier one has read.  From here to the packing below the row is the fp32 path's, bit for bit.
                    const uint2* sb = reinterpret_cast<const uint2*>(reinterpret_cast<const LT*>(sr) + p.V);
                    for (int k0 = 0; k0 < nvec; k0 += 32) {
                        const int k = k0 + lane;
                        float x[4] = {0.0f, 0.0f, 0.0f, 0.0f};
                        if (k < nvec) LV<LT, 4>::get(sb[k], x);
                        __syncwarp();
                        if (k < nvec)
                            sv[k] = make_float4(head * fast_ex2(fmaf(x[0] - fmx, kLog2e, -flz)), head * fast_ex2(fmaf(x[1] - fmx, kLog2e, -flz)),
                                                head * fast_ex2(fmaf(x[2] - fmx, kLog2e, -flz)), head * fast_ex2(fmaf(x[3] - fmx, kLog2e, -flz)));
                    }
                }
                __syncwarp();
                // sr[v] now holds head * y_v: the corrections subtract head * occupancy.  Blank first, then
                // the label columns (a label equal to the blank -- invalid input -- lands on top of it: both kept)
                if (lane == 0) sr[p.blank] = fmaf(-head, gblank, sr[p.blank]);
                __syncwarp();
                const float hz = head * rZ;
                for (int d = lane; d < nd; d += 32) {
                    const int2 e = s_dl[d];
                    const int end = s_dl[d + 1].y;
                    float occ = 0.0f;
                    for (int k = e.y; k < end; ++k) occ += gbuf[k];
                    sr[e.x] = fmaf(-hz, occ, sr[e.x]);
                }
                __syncwarp();
                if constexpr (sizeof(LT) != 4) {
                    // every element rounded once into the lower half: bf16 elements 4k..4k+3 overwrite fp32 elements 2k, 2k+1,
                    // read in this step or an earlier one
                    uint2* so = reinterpret_cast<uint2*>(sr);
                    for (int k0 = 0; k0 < nvec; k0 += 32) {
                        const int k = k0 + lane;
                        float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                        if (k < nvec) v = sv[k];
                        __syncwarp();
                        if (k < nvec) so[k] = make_uint2(bf_pair(v.x, v.y), bf_pair(v.z, v.w));
                    }
                    __syncwarp();
                }
                if (lane == 0) tma_store_1d(grow, sr, (uint32_t)p.V * (uint32_t)sizeof(LT));
                continue;
            } else {
                // wide rows: four vector loads in flight per lane; the blank column is fixed afterwards
                const V_t* xv = reinterpret_cast<const V_t*>(xrow);
                for (int k0 = lane; k0 < nvec; k0 += 128) {
                    V_t xq[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) { const int k = k0 + 32 * u; xq[u] = k < nvec ? __ldg(xv + k) : LV<LT, VEC>::fill(0.0f); }
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int k = k0 + 32 * u;
                        if (k < nvec) {
                            float x[VEC]; LV<LT, VEC>::get(xq[u], x);
                            float y[VEC];
#pragma unroll
                            for (int j = 0; j < VEC; ++j) y[j] = head * fast_ex2(fmaf(x[j] - fmx, kLog2e, -flz));
                            gv[k] = LV<LT, VEC>::pack(y);
                        }
                    }
                }
            }
            for (int v = nvec * VEC + lane; v < p.V; v += 32) {
                float y = fast_ex2(fmaf(ldx(xrow + v) - fmx, kLog2e, -flz));
                if (v == p.blank) y -= gblank;
                stx(grow + v, y * head);
            }
            __syncwarp();
            if (XQ == 0) {
                if (lane == 0 && p.blank < nvec * VEC) {
                    const float y = fast_ex2(fmaf(ldx(xrow + p.blank) - fmx, kLog2e, -flz));
                    stx(grow + p.blank, head * (y - gblank));
                }
                __syncwarp();
            }
            // label columns: one lane per distinct label value sums its run of the rank-ordered
            // occupancies in position order (deterministic, no atomics) and rewrites the column
            for (int d = lane; d < nd; d += 32) {
                const int2 e = s_dl[d];
                const int end = s_dl[d + 1].y;
                float occ = 0.0f;
                for (int k = e.y; k < end; ++k) occ += gbuf[k];
                if (e.x == p.blank) occ += zb;                       // invalid input (label == blank): keep both
                const float y = fast_ex2(fmaf(ldx(xrow + e.x) - fmx, kLog2e, -flz));
                stx(grow + e.x, head * (y - occ * rZ));
            }
        }
    }
    if (STAGED && lane == 0) tma_store_wait_read();      // the rows leave shared memory before the CTA does
    // the stream's next kernel must also see what the walkers write last (loss, loss_sum): one CTA
    // holds this grid open until the walker grid has completed and flushed
    if (blockIdx.x == 0 && blockIdx.y == 0 && tid == 0) asm volatile("griddepcontrol.wait;" ::: "memory");
}

// ---------------------------------------------------------------------------------------
// k_scale_rows: grad[b,t,:] *= head[b] in place.  Row a8 (the operator's Backward: the
// gradient stored by Forward times the head gradient) for callers that ran the fused
// forward+gradient with head = 1.  grid (ceil(T*ceil(V/128)... ) flat over (b, t) rows.
// ---------------------------------------------------------------------------------------
#ifndef CTCB_NO_PLAIN_KERNELS   // non-template kernels: defined in ctcb.cu's translation unit only
__global__ void __launch_bounds__(256) k_scale_rows(float* grad, long long gst_t, long long gst_b, int T, int B, int V,
                                                    const float* head) {
    const int rows_per_cta = 8, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long r = (long long)blockIdx.x * rows_per_cta + warp;
    if (r >= (long long)T * B) return;
    const int b = (int)(r / T), t = (int)(r % T);
    const float h = head[b];
    float* row = grad + b * gst_b + t * gst_t;
    for (int v = lane; v < V; v += 32) row[v] *= h;
}
#endif

// ---------------------------------------------------------------------------------------
// k_greedy_decode: grid B, block 256.  train_ctc_ce.py:149-160 and, with unk >= 0, decode_ctc.py:123-143
// (next-row scope): per frame the best symbol (ties: lowest index) and -- for the <unk> rule -- the second
// best; the symbol of frame j is the best one, or the second best when the best is `unk`; it is kept when
// it differs from the RAW best symbol of frame j-1 (the reference compares against trans[j-1], not against
// the substituted symbol) and is not the blank.
// ---------------------------------------------------------------------------------------
#ifndef CTCB_NO_PLAIN_KERNELS   // non-template kernels: defined in ctcb.cu's translation unit only
// the collapse of frames 0..n-1 by a block of 256 threads: keep[t] = sym[t] != blank && (t == 0 || sym[t] != path[t-1]),
// compacted in order into out[0..len).  Returns len (in every thread); s_scan: 8 ints of shared memory
__device__ __forceinline__ int greedy_collapse(const int* path, const int* sym, int n, int blank, int* out, int* s_scan) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int chunk = (n + 255) / 256;
    const int lo = min(tid * chunk, n), hi = min(lo + chunk, n);
    int cnt = 0;
    for (int t = lo; t < hi; ++t) {
        const int c = sym[t];
        cnt += (c != blank && (t == 0 || c != path[t - 1]));
    }
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
    if (lane == 31) s_scan[warp] = incl;
    __syncthreads();
    int base = 0;
    for (int k = 0; k < warp; ++k) base += s_scan[k];
    int pos = base + incl - cnt;
    for (int t = lo; t < hi; ++t) {
        const int c = sym[t];
        if (c != blank && (t == 0 || c != path[t - 1])) out[pos++] = c;
    }
    int len = 0;
    for (int k = 0; k < 8; ++k) len += s_scan[k];
    return len;
}

template <typename LT = float>
__global__ void __launch_bounds__(256) k_greedy_decode(const LT* logits, long long st_t, long long st_b,
                                                       const void* data_len, int dl_dtype, int T, int B, int V,
                                                       int blank, int unk, int* out_tokens, int* out_len) {
    extern __shared__ int path[];                 // T ints: the raw best symbol; T more: the symbol after the <unk> rule
    __shared__ int s_scan[8];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    long long n64 = data_len ? load_as_int(data_len, dl_dtype, b) : T;
    const int n = (int)(n64 < 0 ? 0 : (n64 > T ? T : n64));
    int* sym = path + T;
    for (int t = warp; t < n; t += 8) {
        const LT* row = logits + b * st_b + t * st_t;
        Top2 tp{-INFINITY, 0x7fffffff, -INFINITY, 0x7fffffff};
        for (int v = lane; v < V; v += 32) top2_push(tp, ldx(row + v), v);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov1 = __shfl_xor_sync(0xffffffffu, tp.v1, o), ov2 = __shfl_xor_sync(0xffffffffu, tp.v2, o);
            const int oi1 = __shfl_xor_sync(0xffffffffu, tp.i1, o), oi2 = __shfl_xor_sync(0xffffffffu, tp.i2, o);
            top2_push(tp, ov1, oi1);
            top2_push(tp, ov2, oi2);
        }
        if (lane == 0) { path[t] = tp.i1; sym[t] = (unk >= 0 && tp.i1 == unk && tp.i2 != 0x7fffffff) ? tp.i2 : tp.i1; }
    }
    __syncthreads();
    const int len = greedy_collapse(path, sym, n, blank, out_tokens + (size_t)b * T, s_scan);
    if (tid == 255) out_len[b] = len;
}

// ---------------------------------------------------------------------------------------
// k_greedy_collapse: grid B, block 256.  The second half of k_greedy_decode for the fused projection's decode epilogue
// (ctcb_proj.cuh, DECODE), which leaves one word per valid frame in out_tokens: the frame's symbol after the <unk> rule,
// bit 31 set when its raw best symbol is `unk`.  An ordinary launch behind the recursion kernel, which may have run beside
// the projection without waiting for it: the utterance's tile flags are acquired here.  tflag == nullptr: an ordinary
// launch right behind the projection (ctcb_proj_greedy_decode, no walkers), stream order is enough.  Writes the
// hypothesis, zeros after it (ctcb_greedy_decode's output on a zeroed buffer) and the length.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_greedy_collapse(const int* tflag, int ntile, const void* data_len, int dl_dtype, int T,
                                                         int blank, int unk, int* out_tokens, int* out_len) {
    extern __shared__ int path[];                 // T ints: the raw best symbol; T more: the symbol after the <unk> rule
    __shared__ int s_scan[8];
    const int b = blockIdx.x, tid = threadIdx.x;
    long long n64 = data_len ? load_as_int(data_len, dl_dtype, b) : T;
    const int n = (int)(n64 < 0 ? 0 : (n64 > T ? T : n64));
    int* sym = path + T;
    for (int k = tid; tflag && k * 128 < n; k += 256) {    // the 128-frame tiles that hold valid frames
        const long long t0 = clock64();           // bounded: a projection that never ran gives garbage, not a hang
        while (ld_acquire_gpu(tflag + (size_t)b * ntile + k) == 0 && clock64() - t0 < kSpinLimit) __nanosleep(256);
    }
    __syncthreads();
    int* row = out_tokens + (size_t)b * T;
    for (int t = tid; t < n; t += 256) {
        const int v = row[t];
        sym[t] = v & 0x7fffffff;
        path[t] = v < 0 ? unk : (v & 0x7fffffff);
    }
    __syncthreads();                              // the row is staged before the hypothesis overwrites it
    const int len = greedy_collapse(path, sym, n, blank, row, s_scan);
    for (int t = len + tid; t < T; t += 256) row[t] = 0;
    if (tid == 255) out_len[b] = len;
}
#endif

// ---------------------------------------------------------------------------------------
// k_edit_distance: grid B, block 128.  scripts/swbd/wer.py:45-68 (next-row scope): Levenshtein
// distance of one (reference, hypothesis) pair per CTA.  Row i of the DP table from row i-1:
//     t[j] = min(d[i-1][j] + 1, d[i-1][j-1] + (ref[i-1] != hyp[j-1]))          (parallel over j)
//     d[i][j] = min(t[j], d[i][j-1] + 1) = j + min_{k<=j}(t[k] - k)            (prefix-min scan)
// each thread owns a contiguous chunk of columns; the scan is a warp shuffle scan of the chunk
// minima plus one hop through shared memory.  (The reference takes d[i-1][j-1] alone on a match;
// neighbouring cells differ by at most one, so the three-way minimum gives the same number.)
// ---------------------------------------------------------------------------------------
#ifndef CTCB_NO_PLAIN_KERNELS   // non-template kernels: defined in ctcb.cu's translation unit only
__global__ void __launch_bounds__(128) k_edit_distance(const int* ref, long long ref_stride, const int* ref_len,
                                                       const int* hyp, long long hyp_stride, const int* hyp_len,
                                                       int max_ref, int max_hyp, int* out_dist, long long* totals) {
    extern __shared__ int esm[];                  // hyp[M], then two rows of M + 1 cells
    __shared__ int s_wmin[4];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int N = min(max(ref_len[b], 0), max_ref), M = min(max(hyp_len[b], 0), max_hyp);
    int* s_hyp = esm; int* row0 = esm + max_hyp; int* row1 = row0 + max_hyp + 1;
    const int* r = ref + b * ref_stride;
    const int* h = hyp + b * hyp_stride;
    for (int j = tid; j < M; j += 128) s_hyp[j] = h[j];
    for (int j = tid; j <= M; j += 128) row0[j] = j;
    __syncthreads();
    const int chunk = (M + 1 + 127) / 128, lo = min(tid * chunk, M + 1), hi = min(lo + chunk, M + 1);
    int* prev = row0; int* cur = row1;
    for (int i = 1; i <= N; ++i) {
        const int ri = r[i - 1];
        int run = INT_MAX;                        // running min of t[k] - k over this thread's chunk
        for (int j = lo; j < hi; ++j) {
            const int t = j == 0 ? i : min(prev[j] + 1, prev[j - 1] + (ri != s_hyp[j - 1]));
            run = min(run, t - j);
            cur[j] = run;                         // chunk-local prefix minimum, completed below
        }
        // exclusive prefix-min of the chunk minima over the block
        int incl = run;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl = min(incl, y); }
        if (lane == 31) s_wmin[warp] = incl;
        int excl = __shfl_up_sync(0xffffffffu, incl, 1);
        if (lane == 0) excl = INT_MAX;
        __syncthreads();
        for (int k = 0; k < warp; ++k) excl = min(excl, s_wmin[k]);
        for (int j = lo; j < hi; ++j) cur[j] = min(cur[j], excl) + j;
        __syncthreads();
        int* sw = prev; prev = cur; cur = sw;
    }
    if (tid == 0) {
        const int d = prev[M];
        out_dist[b] = d;
        if (totals) {
            atomicAdd(reinterpret_cast<unsigned long long*>(totals), (unsigned long long)d);
            atomicAdd(reinterpret_cast<unsigned long long*>(totals + 1), (unsigned long long)N);
        }
    }
}
#endif

}  // namespace ctcb
