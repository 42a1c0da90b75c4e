// ctcb.cu -- host side of libctcb.so: the C ABI declared in include/ctcb.h and
// include/ctcb_dlpack.h.  Validates the problem, carves the caller's workspace, picks the
// walker configuration and enqueues the kernels of ctcb_kernels.cuh on the caller's stream.
// No host synchronisation, no allocation and no CPU arithmetic on the device path.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <new>
#include <utility>
#include <vector>

#include "ctcb.h"
#include "ctcb_dlpack.h"
#include "ctcb_kernels.cuh"
#include "ctcb_meet.cuh"
#include "ctcb_grad2.cuh"
#include "ctcb_proj.cuh"

struct ctcb_mailbox {
    int device = 0, rank = 0, world = 0;
    double* local = nullptr;                       // [2][world][kMailRow] doubles + the counter, cudaMalloc'ed (IPC-exportable)
    void* opened[ctcb::kMailMaxRanks] = {};        // peers' mailboxes mapped by cudaIpcOpenMemHandle
    ctcb::MailboxDev dev{};                        // host copy of the descriptor ...
    ctcb::MailboxDev* dev_d = nullptr;             // ... and where the kernels read it (inside `local`)
    bool connected = false;
};

namespace {

thread_local char g_err[512] = "";
thread_local int g_launches = 0;
thread_local int g_walk_p = 0, g_walk_nw = 0, g_grad_kernel = 0;
struct PendingXchg { struct ctcb_mailbox* mb = nullptr; double* values = nullptr; double* out = nullptr; int count = 0; };
thread_local PendingXchg g_xchg;                      // ctcb_mailbox_exchange_with_next: consumed by the next gradient launch
// enqueues the pending exchange (if any) on `stream`; true when a kernel was launched.  programmatic: as the
// programmatic dependent of the kernel launched just before it (the step's gradient kernel).
bool launch_pending_xchg(cudaStream_t stream, bool programmatic = false) {
    if (!g_xchg.mb) return false;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(1); cfg.blockDim = dim3(32); cfg.dynamicSmemBytes = 0; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = programmatic ? 1 : 0;
    const ctcb::MailboxDev* md = g_xchg.mb->dev_d;
    cudaLaunchKernelEx(&cfg, ctcb::k_mailbox_exchange, md, g_xchg.values, g_xchg.count, g_xchg.out, 0);
    g_xchg = PendingXchg{};
    return true;
}
thread_local const ctcb_proj_t* g_proj = nullptr;      // ctcb_proj_*: the projection whose epilogue replaces k_emit in this call
struct DecodeRequest { int32_t* tokens; int32_t* lengths; int unk; };
thread_local const DecodeRequest* g_decode = nullptr;  // ctcb_proj_forward_decode: the greedy decode the projection's epilogue adds
thread_local bool g_recompute = false;                 // ctcb_proj_forward(keep_for_backward, no logits): the occupancy table follows
thread_local cudaEvent_t* g_prof_events = nullptr;   // when set: one event recorded after every launch
thread_local int g_prof_count = 0;

// ---- tuning / experiment switches -----------------------------------------------------------
// Read from the environment ONCE (CTCB_<NAME>, at first use) and changeable through ctcb_set_option (tests, A/B
// runs): nothing on the per-call host path calls getenv.  -1 = automatic.
enum Opt { OPT_WALK_P, OPT_WALK_NW, OPT_WALK_STAGES, OPT_OVERLAP, OPT_FUSED, OPT_WALK_PER_SM, OPT_EMIT_STAGED,
           OPT_GRAD_STAGED, OPT_MEET, OPT_GRAD2, OPT_GRAD2_BLOCKS, OPT_WALK_HW_WAIT, OPT_GRAD2_OCC, OPT_PROJ_CTAS, OPT_PROJ_DBG, OPT_PROJ_OVERLAP, OPT_MEET_FWD, OPT_WALK_PDL, OPT_GRAD_POLL_NS, OPT_COUNT };
const char* const kOptNames[OPT_COUNT] = {"walk_p", "walk_nw", "walk_stages", "overlap", "fused", "walk_per_sm",
                                          "emit_staged", "grad_staged", "meet", "grad2", "grad2_blocks", "walk_hw_wait", "grad2_occ", "proj_ctas", "proj_dbg", "proj_overlap", "meet_fwd", "walk_pdl", "grad_poll_ns"};
struct Options {
    int v[OPT_COUNT];
    Options() {
        for (int i = 0; i < OPT_COUNT; ++i) {
            char name[64] = "CTCB_";
            size_t k = 5;
            for (const char* c = kOptNames[i]; *c && k + 1 < sizeof(name); ++c) name[k++] = (char)(*c >= 'a' && *c <= 'z' ? *c - 32 : *c);
            name[k] = 0;
            const char* e = getenv(name);
            v[i] = e ? atoi(e) : -1;
        }
    }
};
Options& options() { static Options o; return o; }
inline int opt(Opt i) { return options().v[i]; }

int fail(int code, const char* fmt, ...) {
    va_list ap; va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                   \
    do {                                                                                 \
        cudaError_t e_ = (expr);                                                         \
        if (e_ != cudaSuccess)                                                           \
            return fail(CTCB_EXECUTION_FAILED, "%s: %s", #expr, cudaGetErrorString(e_)); \
    } while (0)

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---- walker configuration -------------------------------------------------------------
struct WalkCfg { int P, NW; };

using WalkFn = void (*)(ctcb::WalkArgs);
struct WalkEntry { int P, NW; WalkFn fn[2][2]; WalkFn fused_bf16[2]; };   // fn[FUSED][HIST]; bf16 logits: fused_bf16[HIST]
#define WALK(P_, NW_) {P_, NW_, {{ctcb::k_walk<P_, NW_, false, false>, ctcb::k_walk<P_, NW_, true, false>}, \
                                 {ctcb::k_walk<P_, NW_, false, true>, ctcb::k_walk<P_, NW_, true, true>}},  \
                                 {ctcb::k_walk<P_, NW_, false, true, ctcb::bf16>, ctcb::k_walk<P_, NW_, true, true, ctcb::bf16>}}
#ifdef CTCB_SMALL_TABLE   // experiment builds: the configurations the BASELINE shapes use
const WalkEntry kWalkTable[] = { WALK(1, 1), WALK(2, 1), WALK(1, 4), WALK(2, 2), WALK(4, 1), WALK(2, 3), WALK(2, 5) };
#else
const WalkEntry kWalkTable[] = {
    WALK(1, 1), WALK(2, 1), WALK(4, 1), WALK(1, 2), WALK(2, 2), WALK(4, 2), WALK(1, 3), WALK(2, 3), WALK(4, 3),
    WALK(1, 4), WALK(2, 4), WALK(4, 4), WALK(2, 5), WALK(2, 6), WALK(1, 8), WALK(2, 8), WALK(4, 8),
    WALK(2, 12), WALK(2, 16), WALK(4, 16),
};
#endif
#undef WALK

const WalkEntry* find_walk(int P, int NW) {
    for (const auto& e : kWalkTable) if (e.P == P && e.NW == NW) return &e;
    return nullptr;
}

// default choice per capacity (pairs = Lmax+1); tuned on B200, see DESIGN.md section 5.
// The choice is part of the workspace layout (history chunks are per walker warp).
const WalkEntry* choose_walk(int pairs) {
    if (opt(OPT_WALK_P) > 0 && opt(OPT_WALK_NW) > 0) {
        const WalkEntry* e = find_walk(opt(OPT_WALK_P), opt(OPT_WALK_NW));
        if (e && e->P * e->NW * 32 >= pairs) return e;
    }
    static const WalkCfg pref[] = {{1, 1}, {2, 1}, {2, 2}, {2, 3}, {2, 4}, {2, 5}, {2, 6}, {2, 8}, {2, 12}, {2, 16}, {4, 16}};
    for (const auto& c : pref)
        if (c.P * c.NW * 32 >= pairs) return find_walk(c.P, c.NW);
    return nullptr;
}

// emission ring depth: as deep as fits a modest budget (several walker CTAs share an SM)
bool pick_stages(int W, int NW, int fused_Lp, int* stages) {
    const size_t budget = 40 * 1024, hard = 200 * 1024;
    for (int s = opt(OPT_WALK_STAGES) > 0 ? opt(OPT_WALK_STAGES) : ctcb::kMaxStages; s >= 2; --s) {
        if (s > ctcb::kMaxStages) continue;
        const size_t need = ctcb::walk_smem_bytes(W, NW, s, fused_Lp);
        if (need <= budget || (s <= 3 && need <= hard)) { *stages = s; return true; }
    }
    return false;
}

// k_grad overlaps k_walk only while every walker CTA of the batch can be resident together.  Fused
// (small-vocabulary) path: the walkers get SMs of their own (shared-memory reservation below).  Wide
// vocabularies: the gradient kernel wants every SM's bandwidth, so the walkers reserve nothing and the
// gradient CTAs share their SMs (measured at cfg3: 238 -> 216 us; with the reservation it was no gain)
bool overlap_allowed(int B, bool fused) {
    if (opt(OPT_OVERLAP) >= 0) return opt(OPT_OVERLAP) != 0;
    (void)fused;
    return B <= 296;
}

// the one-kernel path (k_meet): opt-in / opt-out through the "meet" option, automatic otherwise.  fp32 logits only: a call
// with bf16 logits takes the two-kernel path whatever the option says (k_meet has no bf16 instantiation)
bool meet_wanted(int B) {
    if (opt(OPT_MEET) >= 0) return opt(OPT_MEET) != 0;
    (void)B;
    return false;
}

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) only when a launch needs more than any before it
// (per device and kernel): it is a driver call, and this sits on the per-step host path
cudaError_t ensure_dynamic_smem(const void* fn, size_t bytes) {
    static std::mutex mu;
    static std::vector<std::pair<std::pair<int, const void*>, size_t>> seen;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lk(mu);
    for (auto& e : seen)
        if (e.first.first == dev && e.first.second == fn) {
            if (e.second >= bytes) return cudaSuccess;
            const cudaError_t rc = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
            if (rc == cudaSuccess) e.second = bytes;
            return rc;
        }
    const cudaError_t rc = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (rc == cudaSuccess) seen.push_back({{dev, fn}, bytes});
    return rc;
}

struct Layout {
    size_t off_Tb, off_Lb, off_flags, off_lab, off_rank, off_dl, off_nd, off_fr, off_E, off_hA, off_hB, off_oA, off_oB, off_gprog, off_runv, off_pinfo, off_tflag, off_meet, off_meetlz, off_meetcnt, total;
    int ntile;
    int Lp, W, NB, dense, fused, P, NW;
    int stamp;               // nonzero hash of everything the workspace layout depends on (Workspace::stamp)
    const WalkEntry* walk;
};

// small dense vocabularies: the walkers' own producer warps turn logits rows into emission
// blocks (no k_emit launch, no emission table in HBM)
inline bool fused_emit(int V, int Lmax) {
    (void)Lmax;
    if (opt(OPT_FUSED) == 0) return false;
    return V <= 64;
}

// dense emission table (the whole softmax row, label-indexed by the walkers) when the
// vocabulary is not wider than the label row; gathered columns otherwise
inline bool dense_table(int V, int Lmax) { return V <= Lmax + 1 || V <= 64; }

Layout make_layout(int T, int B, int V, int Lmax, int need_grad) {
    Layout l{};
    l.Lp = (int)align_up((size_t)(Lmax > 0 ? Lmax : 1), 4);
    l.dense = dense_table(V, Lmax) ? 1 : 0;
    l.fused = (l.dense && fused_emit(V, Lmax)) ? 1 : 0;
    l.W = l.dense ? V : Lmax + 1;                 // columns per frame block (64 bytes each)
    l.NB = (T + ctcb::kG - 1) / ctcb::kG;
    l.walk = choose_walk(Lmax + 1);
    l.P = l.walk ? l.walk->P : 1; l.NW = l.walk ? l.walk->NW : 1;
    const size_t pairs = (size_t)l.NW * l.P * 32;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o = align_up(o + bytes, 256); return r; };
    l.off_Tb = take(sizeof(int) * B);
    l.off_Lb = take(sizeof(int) * B);
    l.off_flags = take(sizeof(int) * B);
    l.off_lab = take(sizeof(int) * (size_t)B * l.Lp);
    l.off_rank = take(sizeof(int) * (size_t)B * l.Lp);
    l.off_dl = take(sizeof(int2) * (size_t)B * (l.Lp + 1));
    l.off_nd = take(sizeof(int) * B);
    l.off_gprog = take(sizeof(int) * 4 * (size_t)B);
    l.off_runv = take(sizeof(int2) * 64 * (size_t)B);
    l.off_pinfo = take(sizeof(int2) * (size_t)B);
    l.ntile = (T + 127) / 128 + 1;                // 128-frame tiles of the fused projection (+1: an odd count is paired up)
    l.off_tflag = take(sizeof(int) * (size_t)B * l.ntile);
    l.off_meet = take(sizeof(ctcb::MeetSlot) * (size_t)B * 2 * pairs);      // loss evaluation: walkers that meet in the middle
    l.off_meetlz = take(sizeof(double) * 2 * (size_t)B);
    l.off_meetcnt = take(sizeof(int) * (size_t)B);
    l.off_fr = take(sizeof(float2) * (size_t)B * T);
    l.off_E = take(l.fused ? 0 : sizeof(double) * (size_t)B * l.NB * l.W * ctcb::kEC);
    if (need_grad) {
        l.off_hA = take(sizeof(int2) * (size_t)B * l.NB * ctcb::kG * pairs);
        l.off_hB = take(sizeof(int2) * (size_t)B * l.NB * ctcb::kG * pairs);
        l.off_oA = take(sizeof(int2) * (size_t)B * l.NB * pairs);
        l.off_oB = take(sizeof(int2) * (size_t)B * l.NB * pairs);
    }
    l.total = o;
    unsigned h = 2166136261u;
    for (int v : {T, B, V, Lmax, l.Lp, l.W, l.NB, l.dense, l.fused, l.P, l.NW, need_grad ? 1 : 0}) { h ^= (unsigned)v; h *= 16777619u; }
    l.stamp = (int)(h | 1u);
    return l;
}

ctcb::Workspace carve(const Layout& l, void* ws) {
    char* base = static_cast<char*>(ws);
    ctcb::Workspace w{};
    w.Tb = reinterpret_cast<int*>(base + l.off_Tb);
    w.Lb = reinterpret_cast<int*>(base + l.off_Lb);
    w.flags = reinterpret_cast<int*>(base + l.off_flags);
    w.lab = reinterpret_cast<int*>(base + l.off_lab);
    w.rank = reinterpret_cast<int*>(base + l.off_rank);
    w.dl = reinterpret_cast<int2*>(base + l.off_dl);
    w.nd = reinterpret_cast<int*>(base + l.off_nd);
    w.fr = reinterpret_cast<float2*>(base + l.off_fr);
    w.E = reinterpret_cast<double*>(base + l.off_E);
    w.hA = reinterpret_cast<int2*>(base + l.off_hA);
    w.hB = reinterpret_cast<int2*>(base + l.off_hB);
    w.oA = reinterpret_cast<int2*>(base + l.off_oA);
    w.oB = reinterpret_cast<int2*>(base + l.off_oB);
    w.gprog = reinterpret_cast<int*>(base + l.off_gprog);
    w.runv = reinterpret_cast<int2*>(base + l.off_runv);
    w.pinfo = reinterpret_cast<int2*>(base + l.off_pinfo);
    w.tflag = reinterpret_cast<int*>(base + l.off_tflag); w.ntile = l.ntile;
    w.meet = reinterpret_cast<ctcb::MeetSlot*>(base + l.off_meet);
    w.meetlz = reinterpret_cast<double*>(base + l.off_meetlz);
    w.meetcnt = reinterpret_cast<int*>(base + l.off_meetcnt);
    w.Lp = l.Lp; w.W = l.W; w.NB = l.NB; w.dense = l.dense; w.P = l.P; w.NW = l.NW;
    w.fused = l.fused;
    w.stamp = l.stamp;
    return w;
}

// elements per vector load (VEC is counted in elements; the base must be aligned to VEC * esz bytes)
int pick_vec(const void* base, long long st_t, long long st_b, int V, int esz = 4) {
    auto ok = [&](int v) {
        return V % v == 0 && st_t % v == 0 && st_b % v == 0 && (reinterpret_cast<uintptr_t>(base) % (v * esz)) == 0;
    };
    if (ok(4)) return 4;
    if (ok(2)) return 2;
    return 1;
}
// rows that 1-D bulk copies (TMA) can move: 16-byte aligned row starts and a row of a multiple of 16 bytes.  For fp32 rows
// VEC = 4 already says so; bf16 rows with VEC = 4 are only 8-byte aligned and need the check
bool rows16(const void* base, long long st_t, long long st_b, int V, int esz) {
    return ((long long)V * esz) % 16 == 0 && (st_t * esz) % 16 == 0 && (st_b * esz) % 16 == 0 && reinterpret_cast<uintptr_t>(base) % 16 == 0;
}
inline int dtype_size(int logits_dtype) { return logits_dtype == CTCB_BF16 ? 2 : 4; }

int validate(const ctcb_problem_t* p) {
    if (!p) return fail(CTCB_INVALID_VALUE, "problem is NULL");
    if (p->T <= 0 || p->B <= 0 || p->V <= 1 || p->Lmax < 0)
        return fail(CTCB_INVALID_VALUE, "bad shape T=%d B=%d V=%d Lmax=%d", p->T, p->B, p->V, p->Lmax);
    if (p->blank < 0 || p->blank >= p->V) return fail(CTCB_INVALID_VALUE, "blank %d outside [0,%d)", p->blank, p->V);
    if ((!p->logits && !g_proj) || !p->loss) return fail(CTCB_INVALID_VALUE, "logits and loss must not be NULL");
    if (p->Lmax > 0 && !p->labels) return fail(CTCB_INVALID_VALUE, "labels is NULL");
    auto dt_ok = [](int d) { return d >= CTCB_I32 && d <= CTCB_F64; };
    if (!dt_ok(p->label_dtype) || (p->data_lengths && !dt_ok(p->data_lengths_dtype)) ||
        (p->label_lengths && !dt_ok(p->label_lengths_dtype)))
        return fail(CTCB_INVALID_VALUE, "unsupported label/length dtype");
    if (p->Lmax + 1 > 2048)
        return fail(CTCB_UNSUPPORTED, "Lmax=%d exceeds the supported 2047 labels per utterance", p->Lmax);
    if ((long long)p->B > 65535) return fail(CTCB_UNSUPPORTED, "B=%d exceeds 65535 utterances per call", p->B);
    if (p->logits_row_offsets && !p->data_lengths)
        return fail(CTCB_INVALID_VALUE, "packed logits (logits_row_offsets) need data_lengths");
    return CTCB_OK;
}

ctcb::Problem to_device_problem(const ctcb_problem_t* p) {
    ctcb::Problem d{};
    d.T = p->T; d.B = p->B; d.V = p->V; d.Lmax = p->Lmax; d.blank = p->blank; d.label_pad = p->label_pad;
    d.logits = p->logits; d.st_t = p->logits_stride_t; d.st_b = p->logits_stride_b;
    d.row_off = reinterpret_cast<const long long*>(p->logits_row_offsets);
    d.grad = p->grad; d.gst_t = p->grad_stride_t; d.gst_b = p->grad_stride_b;
    d.labels = p->labels; d.label_dtype = p->label_dtype; d.lst_b = p->label_stride_b; d.lst_l = p->label_stride_l;
    d.data_len = p->data_lengths; d.data_len_dtype = p->data_lengths_dtype;
    d.label_len = p->label_lengths; d.label_len_dtype = p->label_lengths_dtype;
    d.head = p->head_grad; d.loss = p->loss; d.loss_sum = p->loss_sum; d.status = p->status;
    return d;
}

bool is_device_ptr(const void* ptr) {
    if (!ptr) return true;
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, ptr) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}
// the device alias of PINNED host memory (cudaHostAlloc / cudaHostRegister), or nullptr: the 4 B per utterance of the
// loss may be written there by the kernels themselves (ctcb_pipe_submit)
void* pinned_device_alias(const void* ptr) {
    if (!ptr) return nullptr;
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, ptr) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
}

}  // namespace

extern "C" {

int ctcb_version(void) { return CTCB_VERSION; }
const char* ctcb_last_error(void) { return g_err; }
int ctcb_last_launch_count(void) { return g_launches; }
int ctcb_last_walk_config(int32_t* p, int32_t* nw) {
    if (p) *p = g_walk_p;
    if (nw) *nw = g_walk_nw;
    return CTCB_OK;
}

int ctcb_last_grad_kernel(void) { return g_grad_kernel; }

int ctcb_set_option(const char* name, int32_t value) {
    if (!name) return fail(CTCB_INVALID_VALUE, "option name is NULL");
    for (int i = 0; i < OPT_COUNT; ++i)
        if (strcmp(name, kOptNames[i]) == 0) { options().v[i] = value; return CTCB_OK; }
    return fail(CTCB_INVALID_VALUE, "unknown option '%s'", name);
}
int ctcb_get_option(const char* name, int32_t* value) {
    if (!name || !value) return fail(CTCB_INVALID_VALUE, "NULL argument");
    for (int i = 0; i < OPT_COUNT; ++i)
        if (strcmp(name, kOptNames[i]) == 0) { *value = options().v[i]; return CTCB_OK; }
    return fail(CTCB_INVALID_VALUE, "unknown option '%s'", name);
}

int ctcb_workspace_bytes(int32_t T, int32_t B, int32_t V, int32_t Lmax, int32_t need_grad, size_t* out) {
    if (!out) return fail(CTCB_INVALID_VALUE, "out_bytes is NULL");
    if (T <= 0 || B <= 0 || V <= 1 || Lmax < 0) return fail(CTCB_INVALID_VALUE, "bad shape T=%d B=%d V=%d Lmax=%d", T, B, V, Lmax);
    *out = make_layout(T, B, V, Lmax, need_grad).total;
    return CTCB_OK;
}

namespace {

// phase bits
enum { PH_FORWARD = 1, PH_BACKWARD = 2 };

inline void mark(cudaStream_t stream) {
    ++g_launches;
    if (g_prof_events && g_prof_count < 8) cudaEventRecord(g_prof_events[g_prof_count++], stream);
}

// cuTensorMapEncodeTiled through the runtime's driver entry point: libcuda is not linked
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = [] {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q{};
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
            f = nullptr;
        return reinterpret_cast<EncodeTiledFn>(f);
    }();
    return fn;
}

// the projection's operands (hidden, weight, bias): element type, 16-byte strides and bases, device memory
int check_proj_operands(const ctcb_proj_t* pj) {
    if (pj->operand_dtype != CTCB_PROJ_F32 && pj->operand_dtype != CTCB_PROJ_BF16)
        return fail(CTCB_INVALID_VALUE, "projection: operand_dtype %d is neither CTCB_PROJ_F32 nor CTCB_PROJ_BF16", pj->operand_dtype);
    const int per16 = pj->operand_dtype == CTCB_PROJ_BF16 ? 8 : 4;
    if (pj->K % per16 || pj->hidden_stride_t % per16 || pj->hidden_stride_b % per16 || reinterpret_cast<uintptr_t>(pj->hidden) % 16 ||
        reinterpret_cast<uintptr_t>(pj->weight) % 16)
        return fail(CTCB_INVALID_VALUE, "projection: K and the hidden strides must be multiples of 16 bytes, bases 16-byte aligned");
    if (!is_device_ptr(pj->hidden) || !is_device_ptr(pj->weight) || !is_device_ptr(pj->bias))
        return fail(CTCB_INVALID_VALUE, "projection: hidden / weight / bias must be CUDA device memory");
    return CTCB_OK;
}

// the TMA maps of the projection's operands: hidden (K, T, B) in boxes of one 128-byte K block x kPM frames, weight (K, V) in
// boxes of one K block x the CTA's share of a vocabulary tile
int encode_proj_maps(const ctcb_proj_t* pj, int T, int B, int V, int ctas, CUtensorMap* tmA, CUtensorMap* tmB) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return fail(CTCB_UNSUPPORTED, "cuTensorMapEncodeTiled is not available from this driver");
    const bool bf = pj->operand_dtype == CTCB_PROJ_BF16;
    const int esz = bf ? 2 : 4;
    {
        const cuuint64_t gdim[3] = {(cuuint64_t)pj->K, (cuuint64_t)T, (cuuint64_t)B};
        const cuuint64_t gstr[2] = {(cuuint64_t)pj->hidden_stride_t * esz, (cuuint64_t)pj->hidden_stride_b * esz};
        const cuuint32_t box[3] = {(cuuint32_t)(128 / esz), (cuuint32_t)ctcb::kPM, 1};
        const cuuint32_t est[3] = {1, 1, 1};
        const CUresult r = enc(tmA, bf ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(pj->hidden), gdim, gstr, box, est,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(CTCB_INVALID_VALUE, "cuTensorMapEncodeTiled(hidden) failed: %d", (int)r);
    }
    {
        const cuuint64_t gdim[2] = {(cuuint64_t)pj->K, (cuuint64_t)V};
        const cuuint64_t gstr[1] = {(cuuint64_t)pj->K * esz};
        const cuuint32_t box[2] = {(cuuint32_t)(128 / esz), (cuuint32_t)(ctcb::kPN / ctas)};
        const cuuint32_t est[2] = {1, 1};
        const CUresult r = enc(tmB, bf ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(pj->weight), gdim, gstr, box, est,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(CTCB_INVALID_VALUE, "cuTensorMapEncodeTiled(weight) failed: %d", (int)r);
    }
    return CTCB_OK;
}

// the launch fields that depend on the projection alone (the caller adds the problem, workspace and outputs)
ctcb::ProjArgs proj_args(const ctcb_proj_t* pj, int V, int ctas) {
    const int esz = pj->operand_dtype == CTCB_PROJ_BF16 ? 2 : 4;
    ctcb::ProjArgs pa{};
    pa.bias = pj->bias;
    pa.K = pj->K; pa.NT = (V + ctcb::kPN - 1) / ctcb::kPN; pa.KB = (pj->K + 128 / esz - 1) / (128 / esz);
    pa.bf16 = esz == 2 ? 1 : 0;
    pa.ctas = ctas;
    pa.dbg = opt(OPT_PROJ_DBG) > 0 ? opt(OPT_PROJ_DBG) : 0;
    pa.vec4 = (V % 4 == 0 && reinterpret_cast<uintptr_t>(pj->bias) % 16 == 0) ? 1 : 0;
    pa.unk = -1;
    return pa;
}

// CTA pairs (tcgen05 cta_group::2: 256 frames per pair, each CTA stages half of the vocabulary tile) or single CTAs
// (measured: pairs 186 us, single CTAs 190 us per fused forward at cfg3, H = 512)
inline int proj_ctas() { return opt(OPT_PROJ_CTAS) == 1 ? 1 : 2; }

// the projection kernel (ctcb_proj.cuh) in k_emit's place: {row max, normaliser} and the emission table from the
// encoder output, then the metadata CTAs of k_emit (one per utterance)
// beside: the recursion kernel will be launched as the projection's programmatic dependent and follow its tiles (loss
// evaluation only): the metadata kernel then goes FIRST (the walkers poll its "ready" word) and the projection starts beside it
int launch_proj(const ctcb_proj_t* pj, const ctcb_problem_t* p, const ctcb::Problem& dp, const ctcb::Workspace& w,
                const Layout& lay, cudaStream_t stream, bool beside) {
    if (!pj->hidden || !pj->weight || pj->K <= 0) return fail(CTCB_INVALID_VALUE, "projection: hidden / weight is NULL or K <= 0");
    if (lay.fused || lay.dense)
        return fail(CTCB_UNSUPPORTED, "projection fused with the loss needs V > 64 and V > Lmax + 1 (V=%d, Lmax=%d)", p->V, p->Lmax);
    if (p->logits_row_offsets) return fail(CTCB_UNSUPPORTED, "projection: packed logits are not supported");
    if (int rc = check_proj_operands(pj)) return rc;
    const int ctas = proj_ctas();
    const size_t smem = ctcb::proj_smem_bytes(p->Lmax, lay.Lp, p->logits != nullptr, (p->V + ctcb::kPN - 1) / ctcb::kPN, ctas, g_decode != nullptr);
    if (smem > 232448 - 64) return fail(CTCB_UNSUPPORTED, "projection: Lmax=%d label columns do not fit the kernel's shared memory", p->Lmax);
    CUtensorMap tmA, tmB;
    if (int rc = encode_proj_maps(pj, p->T, p->B, p->V, ctas, &tmA, &tmB)) return rc;
    ctcb::ProjArgs pa = proj_args(pj, p->V, ctas);
    pa.p = dp; pa.w = w; pa.logits = const_cast<float*>(p->logits);
    pa.tok = g_decode ? g_decode->tokens : nullptr;
    pa.unk = g_decode ? g_decode->unk : -1;
    // the logits (kept for the gradient kernel) leave through TMA stores when their rows allow a tensor map
    CUtensorMap tmC = tmA;
    pa.store = 0;
    pa.smem_stash = ctcb::proj_smem_stash(p->Lmax, p->logits != nullptr) ? 1 : 0;
    if (p->logits) {
        pa.store = 2;
        if (p->logits_stride_t % 4 == 0 && p->logits_stride_b % 4 == 0 && reinterpret_cast<uintptr_t>(p->logits) % 16 == 0) {
            const cuuint64_t gdim[3] = {(cuuint64_t)p->V, (cuuint64_t)p->T, (cuuint64_t)p->B};
            const cuuint64_t gstr[2] = {(cuuint64_t)p->logits_stride_t * 4, (cuuint64_t)p->logits_stride_b * 4};
            const cuuint32_t box[3] = {32, 32, 1};
            const cuuint32_t est[3] = {1, 1, 1};
            // a (T,B,V) buffer has the batch stride below the frame stride: the map's dimensions stay (V, T, B), strides say the rest
            const CUresult r = encode_tiled()(&tmC, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(p->logits), gdim, gstr, box, est,
                                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r == CUDA_SUCCESS) pa.store = 1;
        }
    }
    const int mtiles = (p->T + ctcb::kPM - 1) / ctcb::kPM;
    const dim3 pgrid(ctas, p->B, (mtiles + ctas - 1) / ctas);
    const int mode = g_decode ? ctcb::kProjLossDecode : ctcb::kProjLoss;
    auto launch_meta = [&](bool programmatic) -> int {
        // per-utterance metadata: k_emit's extra CTA alone (grid.x = 1: every CTA is the metadata CTA)
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(1, p->B); cfg.blockDim = dim3(128); cfg.dynamicSmemBytes = ctcb::emit_smem_bytes(lay.Lp, 0); cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = programmatic ? 1 : 0;
        CUDA_TRY(cudaLaunchKernelEx(&cfg, ctcb::k_emit<1, 0>, dp, w));
        mark(stream);
        return CTCB_OK;
    };
    if (beside) {
        // the tile flags and the metadata-ready words of this call start at zero (one memset: the regions are adjacent)
        CUDA_TRY(cudaMemsetAsync(w.tflag, 0, sizeof(int) * (size_t)p->B * w.ntile, stream));
        CUDA_TRY(cudaMemsetAsync(w.gprog, 0, sizeof(int) * 4 * (size_t)p->B, stream));
        if (int rc = launch_meta(false)) return rc;
        CUDA_TRY(ctcb::launch_proj_emit(tmA, tmB, tmC, pa, mode, pgrid, smem, stream, true));    // programmatic: beside the metadata kernel
        mark(stream);
        return CTCB_OK;
    }
    // decoding: k_greedy_collapse acquires the tile flags, which a previous call on this workspace may have left set
    if (g_decode) CUDA_TRY(cudaMemsetAsync(w.tflag, 0, sizeof(int) * (size_t)p->B * w.ntile, stream));
    CUDA_TRY(ctcb::launch_proj_emit(tmA, tmB, tmC, pa, mode, pgrid, smem, stream, false));
    mark(stream);
    // the metadata kernel as the projection kernel's programmatic dependent -- it starts at once and runs beside it (it
    // reads nothing the projection writes); the recursion kernel that follows is an ordinary launch and waits for both
    if (int rc = launch_meta(!g_prof_events)) return rc;
    return CTCB_OK;
}

// ldt: element type of p->logits and p->grad (CTCB_F32 or CTCB_BF16)
int enqueue(const ctcb_problem_t* p, void* workspace, size_t workspace_bytes, void* stream_, int phases, bool keep_hist,
            int ldt = CTCB_F32) {
    g_grad_kernel = 0;
    if (int rc = validate(p)) return rc;
    if (ldt != CTCB_F32 && ldt != CTCB_BF16)
        return fail(CTCB_INVALID_VALUE, "logits dtype %d is neither CTCB_F32 nor CTCB_BF16 (fp16 logits are not supported)", ldt);
    if (ldt != CTCB_F32 && g_proj) return fail(CTCB_INVALID_VALUE, "the fused projection writes fp32 logits");
    const bool bf = ldt == CTCB_BF16;
    const int esz = dtype_size(ldt);
    const bool need_grad = keep_hist || (phases & PH_BACKWARD);
    if ((phases & PH_BACKWARD) && !p->grad) return fail(CTCB_INVALID_VALUE, "grad is NULL");
    const Layout lay = make_layout(p->T, p->B, p->V, p->Lmax, need_grad);
    if (!workspace) return fail(CTCB_INVALID_VALUE, "workspace is NULL");
    if (workspace_bytes < lay.total)
        return fail(CTCB_WORKSPACE_TOO_SMALL, "workspace %zu < required %zu bytes", workspace_bytes, lay.total);
    if (reinterpret_cast<uintptr_t>(workspace) % 256) return fail(CTCB_INVALID_VALUE, "workspace must be 256-byte aligned");
    if (!is_device_ptr(p->logits) || !(is_device_ptr(p->loss) || pinned_device_alias(p->loss)) || !is_device_ptr(workspace) || !is_device_ptr(p->grad) ||
        !is_device_ptr(p->labels) || !is_device_ptr(p->logits_row_offsets))
        return fail(CTCB_INVALID_VALUE, "logits/labels/loss/grad/workspace must be CUDA device memory (there is no CPU path)");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const ctcb::Problem dp = to_device_problem(p);
    ctcb::Workspace w = carve(lay, workspace);
    w.poll_ns = opt(OPT_GRAD_POLL_NS);

    // ---- the one-kernel path (ctcb_meet.cuh): forward and gradient of small-vocabulary utterances in one CTA each ----
    if (phases == (PH_FORWARD | PH_BACKWARD) && !bf && lay.fused && p->V <= 64 && p->Lmax + 1 <= 128 && meet_wanted(p->B)) {
        const int mp = p->Lmax + 1 <= 32 ? 1 : p->Lmax + 1 <= 64 ? 2 : 4;
        const size_t need = sizeof(int2) * (size_t)p->B * lay.NB * ctcb::kHR * 32 * mp;
        if (lay.off_hA + need <= lay.total) {
            if (p->status) CUDA_TRY(cudaMemsetAsync(p->status, 0, sizeof(int32_t) * (size_t)p->B, stream));
            ctcb::MeetArgs ma{dp, w.hA, lay.NB};
            using MeetFn = void (*)(ctcb::MeetArgs);
            const MeetFn mfn = mp == 1 ? ctcb::k_meet<1> : mp == 2 ? ctcb::k_meet<2> : ctcb::k_meet<4>;
            const size_t msm = ctcb::meet_smem_layout(mp, p->V, lay.Lp).total;
            CUDA_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(mfn), msm));
            g_walk_p = mp; g_walk_nw = 1; g_grad_kernel = 3;
            mfn<<<p->B, 256, msm, stream>>>(ma);
            mark(stream);
            if (launch_pending_xchg(stream)) mark(stream);
            CUDA_TRY(cudaGetLastError());
            return CTCB_OK;
        }
    }
    if (phases & PH_FORWARD) {
        // status words: zeroed here, OR-ed into by the kernels (several CTAs of an utterance report bits)
        if (p->status) CUDA_TRY(cudaMemsetAsync(p->status, 0, sizeof(int32_t) * (size_t)p->B, stream));
        const WalkEntry* we = lay.walk;
        if (!we) return fail(CTCB_UNSUPPORTED, "no walker configuration for Lmax=%d", p->Lmax);
        g_walk_p = we->P; g_walk_nw = we->NW;
        int stages = 0;
        if (!pick_stages(lay.W, we->NW, lay.fused ? lay.Lp : 0, &stages))
            return fail(CTCB_UNSUPPORTED, "Lmax=%d V=%d: the emission ring does not fit in shared memory", p->Lmax, p->V);
        const WalkFn wfn = (bf && lay.fused) ? we->fused_bf16[need_grad ? 1 : 0] : we->fn[lay.fused][need_grad ? 1 : 0];
        size_t smem = ctcb::walk_smem_bytes(lay.W, we->NW, stages, lay.fused ? lay.Lp : 0);
        if (lay.fused && need_grad && (phases & PH_BACKWARD) && overlap_allowed(p->B, true)) {
            // SM partitioning by shared-memory reservation: the gradient kernel runs concurrently
            // (programmatic dependent launch); its CTAs must not share an SM with a walker, whose
            // T-step dependent chain is the critical path.  The walkers therefore ask for all the
            // shared memory their share of an SM has, and the gradient CTAs land on the other SMs.
            int dev = 0, nsm = 148;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
            int per_sm = (2 * p->B + nsm - 1) / nsm;
            // from ~80 utterances on the step is bound by the gradient kernel's throughput, not by the walkers' chain: the
            // walkers are packed four to an SM and the gradient CTAs get the other SMs while the walkers run
            // (scripts/regime_sweep.py: B = 96 89.8 -> 80.2 us, 128 113.5 -> 102.6, 148 126.4 -> 111.8)
            if (p->B >= 80 && per_sm < 4) per_sm = 4;
            if (opt(OPT_WALK_PER_SM) > 0) per_sm = opt(OPT_WALK_PER_SM) > (2 * p->B + nsm - 1) / nsm ? opt(OPT_WALK_PER_SM) : (2 * p->B + nsm - 1) / nsm;
            const size_t share = (size_t)233472 / per_sm;
            size_t want = share > 2048 ? (share - 1024) / 128 * 128 : 0;
            cudaFuncAttributes fa{};
            CUDA_TRY(cudaFuncGetAttributes(&fa, reinterpret_cast<const void*>(wfn)));
            const size_t cap = 232448 - (fa.sharedSizeBytes + 127) / 128 * 128;   // opt-in maximum minus the kernel's static part
            if (want > cap) want = cap;
            if (want > smem) smem = want;
        }
        const int vec = pick_vec(p->logits, p->logits_stride_t, p->logits_row_offsets ? 0 : p->logits_stride_b, p->V, esz);
        CUDA_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(wfn), smem));
        // NQ: vector loads per lane that hold one logits row in registers (0 = two-pass)
        const int units = (p->V / vec + 31) / 32;
        int nq = units <= 1 ? 1 : units <= 2 ? 2 : units <= 4 ? 4 : units <= 8 ? 8 : units <= 16 ? 16 : 0;
        // wide vocabularies with 16-byte aligned rows: the frame block's rows staged in shared memory by bulk copies
        // (bf16 rows: also V * 2 a multiple of 16 bytes and 16-byte aligned rows)
        const bool staged = !lay.fused && vec == 4 && (nq == 0 || nq >= 8) && ctcb::emit_smem_bytes(lay.Lp, p->V) <= 75 * 1024 &&
                            opt(OPT_EMIT_STAGED) != 0 &&
                            rows16(p->logits, p->logits_stride_t, p->logits_row_offsets ? 0 : p->logits_stride_b, p->V, esz);
        if (staged) nq = -1;
        auto launch_emit = [&]() -> int {
            const int bpc = ctcb::emit_blocks_per_cta(nq);
            const int nblk = (lay.NB + bpc - 1) / bpc + 1;          // + the metadata CTA of each utterance
            const dim3 egrid(nblk, p->B);
            const size_t esm = ctcb::emit_smem_bytes(lay.Lp, staged ? p->V : 0);
            if (staged) {
                auto efn = bf ? ctcb::k_emit<4, -1, ctcb::bf16> : ctcb::k_emit<4, -1>;
                if (esm > 48 * 1024) CUDA_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(efn), esm));
                efn<<<egrid, 256, esm, stream>>>(dp, w);
            } else {
#define EMIT_LAUNCH(V_, Q_) (bf ? ctcb::k_emit<V_, Q_, ctcb::bf16> : ctcb::k_emit<V_, Q_>)<<<egrid, 128, esm, stream>>>(dp, w)
#define EMIT_NQ(V_) switch (nq) { case 1: EMIT_LAUNCH(V_, 1); break; case 2: EMIT_LAUNCH(V_, 2); break; \
                                  case 4: EMIT_LAUNCH(V_, 4); break; case 8: EMIT_LAUNCH(V_, 8); break;  \
                                  case 16: EMIT_LAUNCH(V_, 16); break; default: EMIT_LAUNCH(V_, 0); break; }
                switch (vec) {
                    case 4: EMIT_NQ(4); break;
                    case 2: EMIT_NQ(2); break;
                    default: EMIT_NQ(1); break;
                }
#undef EMIT_NQ
#undef EMIT_LAUNCH
            }
            mark(stream);
            return CTCB_OK;
        };
        // ctcb_mailbox_exchange_with_next on a forward-only call: the exchange kernel goes first and the recursion
        // kernel is its programmatic dependent -- it starts while the exchange's one warp talks to the peers.
        // (With a gradient kernel in the call the exchange goes behind that one instead, see below.)
        const bool xchg = !(phases & PH_BACKWARD) && launch_pending_xchg(stream);
        if (xchg) mark(stream);
        // loss evaluation from the encoder output: the recursion kernel is the projection's programmatic dependent and
        // follows its 128-frame tiles (the utterances' first tiles are scheduled first) instead of waiting for the kernel
        const bool beside = g_proj && !need_grad && !xchg && !g_prof_events && opt(OPT_PROJ_OVERLAP) != 0;
        // loss evaluation (no history): the alpha and the beta walker take half of the frames each and meet in the middle --
        // while every walker CTA of the batch can be resident at once (beyond that one walker per utterance does less work:
        // cfg5, B = 1024: 136 us against 153).  Beside the projection kernel one walker per utterance is the better schedule
        // (the walkers share the few SMs the projection leaves free: 163 us against 168 with twice as many walker CTAs,
        // also when the tiles were computed from both ends inwards -- that tile order was measured and removed).
        const bool meet_fwd = !need_grad && (opt(OPT_MEET_FWD) >= 0 ? opt(OPT_MEET_FWD) != 0 : (p->B <= 148 && !beside));
        if (meet_fwd) CUDA_TRY(cudaMemsetAsync(w.meetcnt, 0, sizeof(int) * (size_t)p->B, stream));
        auto launch_walk = [&](bool after_xchg, bool beside_proj) -> int {
            ctcb::WalkArgs wa{dp, w, p->T, stages, p->blank, p->loss, p->loss_sum, nullptr, 0, 1, 0, 0, 0};
            wa.beside_proj = beside_proj ? 1 : 0;
            // the fused recursion kernel behind whatever the stream holds (the previous step's gradient kernel in a training
            // loop's graph): launched programmatically, its CTAs become resident during that kernel's tail and wait there
            const bool pdl = lay.fused && !after_xchg && !beside_proj && opt(OPT_WALK_PDL) != 0;
            wa.pdl_wait = pdl ? 1 : 0;
            wa.meet = meet_fwd ? 1 : 0;
            // several walker CTAs per SM: the producers wait in hardware (no polling instructions)
            wa.hw_wait = opt(OPT_WALK_HW_WAIT) >= 0 ? opt(OPT_WALK_HW_WAIT) : (2 * p->B > 148 ? 1 : 0);
            // the per-group progress is for gradient CTAs that run concurrently with the walkers; a gradient kernel that
            // runs afterwards polls the same words once, so the final count is enough
            wa.publish = ((phases & PH_BACKWARD) && !g_prof_events && overlap_allowed(p->B, lay.fused != 0)) ? 1 : 2;
            const int wthreads = (we->NW + (lay.fused ? ctcb::kFusedProducers + 1 : 1)) * 32;
            cudaLaunchConfig_t cfg{};
            cfg.gridDim = dim3(p->B, (need_grad || meet_fwd) ? 2 : 1); cfg.blockDim = dim3(wthreads); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            attr[0].val.programmaticStreamSerializationAllowed = 1;
            cfg.attrs = attr; cfg.numAttrs = (after_xchg || pdl) ? 1 : 0;
            CUDA_TRY(cudaLaunchKernelEx(&cfg, wfn, wa));
            mark(stream);
            return CTCB_OK;
        };
        if (g_proj) {
            if (int rc = launch_proj(g_proj, p, dp, w, lay, stream, beside)) return rc;
        } else if (!lay.fused) { if (int rc = launch_emit()) return rc; }
        if (int rc = launch_walk((xchg && lay.fused != 0) || beside, beside)) return rc;
        if (g_recompute) {
            // the recomputing training forward: the history becomes the occupancy table O that ctcb_proj_backward reads
            CUDA_TRY(ctcb::launch_proj_occ(dp, w, stream));
            mark(stream);
        }
        if (g_decode) {
            // the hypotheses from the projection's per-frame words (an ordinary launch: it acquires the tile flags itself)
            const size_t dsm = 2 * sizeof(int) * (size_t)p->T;
            if (dsm > 48 * 1024) CUDA_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(ctcb::k_greedy_collapse), dsm));
            ctcb::k_greedy_collapse<<<p->B, 256, dsm, stream>>>(w.tflag, w.ntile, p->data_lengths, p->data_lengths_dtype, p->T, p->blank,
                                                                g_decode->unk, g_decode->tokens, g_decode->lengths);
            mark(stream);
        }
    }
    if (phases & PH_BACKWARD) {
        ctcb::GradArgs ga{dp, w};
        const int gpairs = p->Lmax + 1;
        const int gch = gpairs <= 32 ? 1 : gpairs <= 64 ? 2 : gpairs <= 128 ? 4 : gpairs <= 256 ? 8 : gpairs <= 512 ? 16 : 0;
        size_t gsm = ctcb::grad_smem_bytes(lay.Lp, 32 * gch);
        int gthreads = 128;
        if (gsm > 200 * 1024) return fail(CTCB_UNSUPPORTED, "Lmax=%d too long for the gradient kernel", p->Lmax);
        int vec = pick_vec(p->logits, p->logits_stride_t, p->logits_row_offsets ? 0 : p->logits_stride_b, p->V, esz);
        const int gvec = pick_vec(p->grad, p->grad_stride_t, p->grad_stride_b, p->V, esz);
        if (gvec < vec) vec = gvec;
        const int ch = gch;
        const int units = (p->V / vec + 31) / 32;
        const int xq = units <= 1 ? 1 : units <= 2 ? 2 : units <= 4 ? 4 : 0;
        const dim3 ggrid(p->B, lay.NB);                  // one frame block per CTA, utterance-fastest
        using GradFn = void (*)(ctcb::GradArgs);
        GradFn gfn = nullptr;
#define GRAD_X(V_, C_, T_) (xq == 1 ? ctcb::k_grad<V_, C_, 1, 0, T_> : xq == 2 ? ctcb::k_grad<V_, C_, 2, 0, T_> : \
                            xq == 4 ? ctcb::k_grad<V_, C_, 4, 0, T_> : ctcb::k_grad<V_, C_, 0, 0, T_>)
#define GRAD_CH(V_, T_) (ch == 1 ? GRAD_X(V_, 1, T_) : ch == 2 ? GRAD_X(V_, 2, T_) : ch == 4 ? GRAD_X(V_, 4, T_) : ch == 8 ? GRAD_X(V_, 8, T_) : \
                         ch == 16 ? GRAD_X(V_, 16, T_) : GRAD_X(V_, 0, T_))
        if (bf) gfn = vec == 4 ? GRAD_CH(4, ctcb::bf16) : vec == 2 ? GRAD_CH(2, ctcb::bf16) : GRAD_CH(1, ctcb::bf16);
        else    gfn = vec == 4 ? GRAD_CH(4, float) : vec == 2 ? GRAD_CH(2, float) : GRAD_CH(1, float);
#undef GRAD_CH
#undef GRAD_X
        // batches that run after the walkers (no overlap): the high-occupancy variant of the register-resident kernels
        if (ch >= 1 && ch <= 4 && !((phases & PH_FORWARD) && !g_prof_events && overlap_allowed(p->B, lay.fused != 0))) {
#define GRADO_X(V_, C_, T_) (xq == 1 ? ctcb::k_grad<V_, C_, 1, 1, T_> : xq == 2 ? ctcb::k_grad<V_, C_, 2, 1, T_> : \
                             xq == 4 ? ctcb::k_grad<V_, C_, 4, 1, T_> : ctcb::k_grad<V_, C_, 0, 1, T_>)
#define GRADO_CH(V_, T_) (ch == 1 ? GRADO_X(V_, 1, T_) : ch == 2 ? GRADO_X(V_, 2, T_) : GRADO_X(V_, 4, T_))
            if (bf) gfn = vec == 4 ? GRADO_CH(4, ctcb::bf16) : vec == 2 ? GRADO_CH(2, ctcb::bf16) : GRADO_CH(1, ctcb::bf16);
            else    gfn = vec == 4 ? GRADO_CH(4, float) : vec == 2 ? GRADO_CH(2, float) : GRADO_CH(1, float);
#undef GRADO_CH
#undef GRADO_X
        }
        bool grad2 = false;
        // small vocabularies (fused path): the gradient kernel that normalises by P(l|x) (ctcb_grad2.cuh)
        // (measured, scripts/grad2_blocks_sweep.py: from 64 utterances on it wins -- 13 % at B = 128 and 1024, 21 % at 256;
        // below that the step is the walkers' chain plus the gradient kernel's tail, where k_grad is a little shorter)
        const bool want_grad2 = opt(OPT_GRAD2) >= 0 ? opt(OPT_GRAD2) != 0 : (p->B >= 64 && ch <= 4);
        if (lay.fused && p->V <= 64 && ch >= 1 && want_grad2) {
            // two register budgets (profiles/r3e_*, r3f_*): 80 registers / 6 CTAs per SM while the walkers run beside the
            // kernel, 72 registers / 7 CTAs per SM for batches whose gradient kernel runs after the walkers
            bool occ = (phases & PH_FORWARD) && !g_prof_events && overlap_allowed(p->B, true);
            if (opt(OPT_GRAD2_OCC) >= 0) occ = opt(OPT_GRAD2_OCC) != 0;
#define GRAD2_O(V_, C_, T_) (occ ? ctcb::k_grad2<V_, C_, 1, T_> : ctcb::k_grad2<V_, C_, 0, T_>)
#define GRAD2_CH(V_, T_) (ch == 1 ? GRAD2_O(V_, 1, T_) : ch == 2 ? GRAD2_O(V_, 2, T_) : ch == 4 ? GRAD2_O(V_, 4, T_) : \
                          ch == 8 ? GRAD2_O(V_, 8, T_) : GRAD2_O(V_, 16, T_))
            if (bf) gfn = vec == 4 ? GRAD2_CH(4, ctcb::bf16) : vec == 2 ? GRAD2_CH(2, ctcb::bf16) : GRAD2_CH(1, ctcb::bf16);
            else    gfn = vec == 4 ? GRAD2_CH(4, float) : vec == 2 ? GRAD2_CH(2, float) : GRAD2_CH(1, float);
#undef GRAD2_CH
#undef GRAD2_O
            gsm = ctcb::grad2_smem_bytes(ch);
            grad2 = true;
        }
        // wide vocabularies with 16-byte aligned rows: the frame block's rows staged in shared memory by bulk copies
        const size_t gsm_staged = ctcb::grad_smem_bytes(lay.Lp, 32 * gch, p->V);
        // (bf16 rows: also V * 2 a multiple of 16 bytes and 16-byte aligned rows, logits and gradient)
        if (xq == 0 && vec == 4 && gsm_staged <= 75 * 1024 && opt(OPT_GRAD_STAGED) != 0 &&
            rows16(p->logits, p->logits_stride_t, p->logits_row_offsets ? 0 : p->logits_stride_b, p->V, esz) &&
            rows16(p->grad, p->grad_stride_t, p->grad_stride_b, p->V, esz)) {
#define GRAD_ST(T_) (ch == 1 ? ctcb::k_grad<4, 1, -1, 0, T_> : ch == 2 ? ctcb::k_grad<4, 2, -1, 0, T_> : ch == 4 ? ctcb::k_grad<4, 4, -1, 0, T_> : \
                     ch == 8 ? ctcb::k_grad<4, 8, -1, 0, T_> : ch == 16 ? ctcb::k_grad<4, 16, -1, 0, T_> : ctcb::k_grad<4, 0, -1, 0, T_>)
            gfn = bf ? GRAD_ST(ctcb::bf16) : GRAD_ST(float);
#undef GRAD_ST
            gsm = gsm_staged;
            gthreads = 256;                      // 8 warps, one frame each
        }
        if (gsm > 48 * 1024) CUDA_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(gfn), gsm));
        // programmatic dependent of k_walk when both are enqueued by this call: the gradient CTAs
        // start while the walkers run and wait per frame block on Workspace::gprog.  Not when
        // per-kernel events sit between the launches (ctcb_loss_grad_timed) or for batches whose
        // walkers do not fit the GPU at once (the waiting CTAs would hold slots the walkers need).
        const bool overlap = (phases & PH_FORWARD) && !g_prof_events && overlap_allowed(p->B, lay.fused != 0);
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = ggrid; cfg.blockDim = dim3(gthreads); cfg.dynamicSmemBytes = gsm; cfg.stream = stream;
        if (grad2) {
            // k_grad2: a CTA takes several consecutive frame blocks (metadata and P(l|x) once per CTA)
            const int gb = opt(OPT_GRAD2_BLOCKS) > 0 ? opt(OPT_GRAD2_BLOCKS) : 4;      // one whole frame block per warp
            cfg.gridDim = dim3(p->B, (lay.NB + gb - 1) / gb);
        }
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = overlap ? 1 : 0;
        CUDA_TRY(cudaLaunchKernelEx(&cfg, gfn, ga));
        g_grad_kernel = grad2 ? 2 : 1;
        mark(stream);
        // ctcb_mailbox_exchange_with_next: behind the gradient kernel, as its programmatic dependent
        if (launch_pending_xchg(stream, true)) mark(stream);
    }
    CUDA_TRY(cudaGetLastError());
    return CTCB_OK;
}

}  // namespace

int ctcb_loss_grad(const ctcb_problem_t* p, void* workspace, size_t workspace_bytes, void* stream) {
    return ctcb_loss_grad_typed(p, CTCB_F32, workspace, workspace_bytes, stream);
}

int ctcb_loss_grad_typed(const ctcb_problem_t* p, int32_t logits_dtype, void* workspace, size_t workspace_bytes, void* stream) {
    g_launches = 0;
    const bool need_grad = p && p->grad != nullptr;
    return enqueue(p, workspace, workspace_bytes, stream, need_grad ? (PH_FORWARD | PH_BACKWARD) : PH_FORWARD, need_grad, logits_dtype);
}

int ctcb_loss_grad_timed(const ctcb_problem_t* p, void* workspace, size_t workspace_bytes, void* stream_,
                         float* kernel_ms, int32_t* n_kernels) {
    if (!kernel_ms || !n_kernels) return fail(CTCB_INVALID_VALUE, "kernel_ms / n_kernels is NULL");
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    cudaEvent_t ev[9];
    for (auto& e : ev) CUDA_TRY(cudaEventCreate(&e));
    CUDA_TRY(cudaEventRecord(ev[0], stream));
    g_prof_events = ev + 1; g_prof_count = 0;
    const int rc = ctcb_loss_grad(p, workspace, workspace_bytes, stream);
    const int n = g_prof_count;
    g_prof_events = nullptr; g_prof_count = 0;
    if (rc == CTCB_OK) {
        CUDA_TRY(cudaStreamSynchronize(stream));
        for (int i = 0; i < n; ++i) CUDA_TRY(cudaEventElapsedTime(&kernel_ms[i], ev[i], ev[i + 1]));
        *n_kernels = n;
    }
    for (auto& e : ev) cudaEventDestroy(e);
    return rc;
}

int ctcb_forward(const ctcb_problem_t* p, int32_t keep_for_backward, void* workspace, size_t workspace_bytes, void* stream) {
    return ctcb_forward_typed(p, CTCB_F32, keep_for_backward, workspace, workspace_bytes, stream);
}

int ctcb_forward_typed(const ctcb_problem_t* p, int32_t logits_dtype, int32_t keep_for_backward, void* workspace,
                       size_t workspace_bytes, void* stream) {
    g_launches = 0;
    return enqueue(p, workspace, workspace_bytes, stream, PH_FORWARD, keep_for_backward != 0, logits_dtype);
}

int ctcb_backward(const ctcb_problem_t* p, void* workspace, size_t workspace_bytes, void* stream) {
    return ctcb_backward_typed(p, CTCB_F32, workspace, workspace_bytes, stream);
}

int ctcb_backward_typed(const ctcb_problem_t* p, int32_t logits_dtype, void* workspace, size_t workspace_bytes, void* stream) {
    g_launches = 0;
    return enqueue(p, workspace, workspace_bytes, stream, PH_BACKWARD, true, logits_dtype);
}

int ctcb_proj_forward(const ctcb_proj_t* proj, const ctcb_problem_t* p, int32_t keep_for_backward, void* workspace,
                      size_t workspace_bytes, void* stream) {
    if (!proj) return fail(CTCB_INVALID_VALUE, "proj is NULL");
    g_launches = 0;
    g_proj = proj;
    // keep_for_backward without a logits buffer: the history is kept and turned into the occupancy table, the logits are
    // never stored, and ctcb_proj_backward forms the product again
    g_recompute = keep_for_backward && p && !p->logits;
    const int rc = enqueue(p, workspace, workspace_bytes, stream, PH_FORWARD, keep_for_backward != 0);
    g_proj = nullptr;
    g_recompute = false;
    return rc;
}

int ctcb_proj_forward_decode(const ctcb_proj_t* proj, const ctcb_problem_t* p, int32_t keep_for_backward, int32_t unk,
                             int32_t* out_tokens, int32_t* out_lengths, void* workspace, size_t workspace_bytes, void* stream) {
    if (!out_tokens || !out_lengths) return fail(CTCB_INVALID_VALUE, "NULL argument");
    if (p && unk >= p->V) return fail(CTCB_INVALID_VALUE, "unk %d outside the vocabulary (V=%d; -1 = no <unk> rule)", unk, p->V);
    if (p && p->T > 0 && 2 * sizeof(int) * (size_t)p->T > 200 * 1024) return fail(CTCB_UNSUPPORTED, "T=%d too long for the decode kernel", p->T);
    if (!is_device_ptr(out_tokens) || !is_device_ptr(out_lengths)) return fail(CTCB_INVALID_VALUE, "buffers must be CUDA device memory");
    const DecodeRequest req{out_tokens, out_lengths, unk < 0 ? -1 : unk};
    g_decode = &req;
    const int rc = ctcb_proj_forward(proj, p, keep_for_backward, workspace, workspace_bytes, stream);
    g_decode = nullptr;
    return rc;
}

int ctcb_proj_greedy_decode(const ctcb_proj_t* proj, int32_t T, int32_t B, int32_t V, const void* data_lengths,
                            int32_t data_lengths_dtype, int32_t blank, int32_t unk, int32_t* out_tokens, int32_t* out_lengths,
                            void* stream) {
    g_launches = 0;
    if (!proj || !out_tokens || !out_lengths) return fail(CTCB_INVALID_VALUE, "NULL argument");
    if (T <= 0 || B <= 0 || V <= 0) return fail(CTCB_INVALID_VALUE, "bad shape");
    if (unk >= V) return fail(CTCB_INVALID_VALUE, "unk %d outside the vocabulary (V=%d; -1 = no <unk> rule)", unk, V);
    if (data_lengths && (data_lengths_dtype < CTCB_I32 || data_lengths_dtype > CTCB_F64))
        return fail(CTCB_INVALID_VALUE, "unsupported length dtype %d", data_lengths_dtype);
    const size_t dsm = 2 * sizeof(int) * (size_t)T;
    if (dsm > 200 * 1024) return fail(CTCB_UNSUPPORTED, "T=%d too long for the decode kernel", T);
    if (!proj->hidden || !proj->weight || proj->K <= 0) return fail(CTCB_INVALID_VALUE, "projection: hidden / weight is NULL or K <= 0");
    if (int rc = check_proj_operands(proj)) return rc;
    if (!is_device_ptr(out_tokens) || !is_device_ptr(out_lengths) || !is_device_ptr(data_lengths))
        return fail(CTCB_INVALID_VALUE, "buffers must be CUDA device memory");
    const int ctas = proj_ctas();
    const int NT = (V + ctcb::kPN - 1) / ctcb::kPN;
    CUtensorMap tmA, tmB;
    if (int rc = encode_proj_maps(proj, T, B, V, ctas, &tmA, &tmB)) return rc;
    // no labels and no workspace: of the problem the decode-only epilogue reads the shape and the frame counts
    ctcb::ProjArgs pa = proj_args(proj, V, ctas);
    pa.p.T = T; pa.p.B = B; pa.p.V = V; pa.p.blank = blank;
    pa.p.data_len = data_lengths; pa.p.data_len_dtype = data_lengths_dtype;
    pa.tok = out_tokens;
    pa.unk = unk < 0 ? -1 : unk;
    const int mtiles = (T + ctcb::kPM - 1) / ctcb::kPM;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CUDA_TRY(ctcb::launch_proj_emit(tmA, tmB, tmA, pa, ctcb::kProjDecode, dim3(ctas, B, (mtiles + ctas - 1) / ctas),
                                    ctcb::proj_smem_bytes(0, 0, false, NT, ctas, true), st, false));
    mark(st);
    // the collapse right behind the projection: stream order, no tile flags
    if (dsm > 48 * 1024) CUDA_TRY(ensure_dynamic_smem(reinterpret_cast<const void*>(ctcb::k_greedy_collapse), dsm));
    ctcb::k_greedy_collapse<<<B, 256, dsm, st>>>(nullptr, 0, data_lengths, data_lengths_dtype, T, blank, pa.unk, out_tokens, out_lengths);
    CUDA_TRY(cudaGetLastError());
    mark(st);
    return CTCB_OK;
}

int ctcb_proj_loss_grad(const ctcb_proj_t* proj, const ctcb_problem_t* p, void* workspace, size_t workspace_bytes, void* stream) {
    if (!proj) return fail(CTCB_INVALID_VALUE, "proj is NULL");
    if (p && (!p->logits || !p->grad)) return fail(CTCB_INVALID_VALUE, "ctcb_proj_loss_grad needs p->logits and p->grad");
    g_launches = 0;
    g_proj = proj;
    const int rc = enqueue(p, workspace, workspace_bytes, stream, PH_FORWARD | PH_BACKWARD, true);
    g_proj = nullptr;
    return rc;
}

int ctcb_proj_backward(const ctcb_proj_t* proj, const ctcb_problem_t* p, void* workspace, size_t workspace_bytes, void* stream_) {
    g_launches = 0;
    if (!proj) return fail(CTCB_INVALID_VALUE, "proj is NULL");
    g_proj = proj;                                  // validate: the logits pointer is not needed
    const int vrc = validate(p);
    g_proj = nullptr;
    if (vrc) return vrc;
    if (!p->grad) return fail(CTCB_INVALID_VALUE, "grad is NULL");
    const Layout lay = make_layout(p->T, p->B, p->V, p->Lmax, 1);
    if (lay.fused || lay.dense)
        return fail(CTCB_UNSUPPORTED, "projection fused with the loss needs V > 64 and V > Lmax + 1 (V=%d, Lmax=%d)", p->V, p->Lmax);
    if (p->logits_row_offsets) return fail(CTCB_UNSUPPORTED, "projection: packed logits are not supported");
    if (!workspace) return fail(CTCB_INVALID_VALUE, "workspace is NULL");
    if (workspace_bytes < lay.total)
        return fail(CTCB_WORKSPACE_TOO_SMALL, "workspace %zu < required %zu bytes", workspace_bytes, lay.total);
    if (reinterpret_cast<uintptr_t>(workspace) % 256) return fail(CTCB_INVALID_VALUE, "workspace must be 256-byte aligned");
    if (!is_device_ptr(workspace) || !is_device_ptr(p->grad) || !is_device_ptr(p->labels) || !is_device_ptr(p->head_grad))
        return fail(CTCB_INVALID_VALUE, "labels/grad/head_grad/workspace must be CUDA device memory (there is no CPU path)");
    if (!proj->hidden || !proj->weight || proj->K <= 0) return fail(CTCB_INVALID_VALUE, "projection: hidden / weight is NULL or K <= 0");
    if (int rc = check_proj_operands(proj)) return rc;
    const int ctas = proj_ctas();
    const int NT = (p->V + ctcb::kPN - 1) / ctcb::kPN;
    const size_t smem = ctcb::proj_smem_bytes(p->Lmax, lay.Lp, true, NT, ctas);
    if (smem > 232448 - 64) return fail(CTCB_UNSUPPORTED, "projection: Lmax=%d label columns do not fit the kernel's shared memory", p->Lmax);
    CUtensorMap tmA, tmB;
    if (int rc = encode_proj_maps(proj, p->T, p->B, p->V, ctas, &tmA, &tmB)) return rc;
    ctcb::ProjArgs pa = proj_args(proj, p->V, ctas);
    pa.p = to_device_problem(p);
    pa.w = carve(lay, workspace);
    // G leaves through TMA tile stores when its rows allow a tensor map, else as coalesced rows from the staging tiles
    CUtensorMap tmC = tmA;
    pa.store = 2;
    if (p->grad_stride_t % 4 == 0 && p->grad_stride_b % 4 == 0 && reinterpret_cast<uintptr_t>(p->grad) % 16 == 0) {
        const cuuint64_t gdim[3] = {(cuuint64_t)p->V, (cuuint64_t)p->T, (cuuint64_t)p->B};
        const cuuint64_t gstr[2] = {(cuuint64_t)p->grad_stride_t * 4, (cuuint64_t)p->grad_stride_b * 4};
        const cuuint32_t box[3] = {32, 32, 1};
        const cuuint32_t est[3] = {1, 1, 1};
        const CUresult r = encode_tiled()(&tmC, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, p->grad, gdim, gstr, box, est,
                                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r == CUDA_SUCCESS) pa.store = 1;
    }
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    const int mtiles = (p->T + ctcb::kPM - 1) / ctcb::kPM;
    CUDA_TRY(ctcb::launch_proj_emit(tmA, tmB, tmC, pa, ctcb::kProjGrad, dim3(ctas, p->B, (mtiles + ctas - 1) / ctas), smem, stream, false));
    mark(stream);
    return CTCB_OK;
}

// ---- host-buffer entry ------------------------------------------------------------------
namespace {
struct HostScratch {
    void* ptr = nullptr; size_t bytes = 0;
    cudaStream_t stream = nullptr;
};
std::mutex g_hs_mu;
HostScratch g_hs[64];
size_t dt_size(int d) { return (d == CTCB_I32 || d == CTCB_F32) ? 4 : 8; }
}  // namespace

namespace {
int loss_grad_host_impl(const ctcb_problem_t* hp, int device, float** dev_grad);

long long host_len(const void* p, int dtype, int b) {
    switch (dtype) {
        case CTCB_I32: return static_cast<const int32_t*>(p)[b];
        case CTCB_I64: return static_cast<const int64_t*>(p)[b];
        case CTCB_F32: return (long long)static_cast<const float*>(p)[b];
        default: return (long long)static_cast<const double*>(p)[b];
    }
}
// Host entries, packed logits (ctcb_problem_t.logits_row_offsets, HOST arrays here): bytes of the buffer =
// max_b (offset_b + T_b * V) floats.  Utterance-major rows only (logits_stride_t == V).
int packed_logits_bytes(const ctcb_problem_t* hp, size_t* bytes) {
    if (hp->logits_stride_t != hp->V) return fail(CTCB_INVALID_VALUE, "packed logits need logits_stride_t == V");
    long long hi = 0;
    for (int b = 0; b < hp->B; ++b) {
        long long t = host_len(hp->data_lengths, hp->data_lengths_dtype, b);
        t = t < 0 ? 0 : (t > hp->T ? hp->T : t);
        const long long off = hp->logits_row_offsets[b];
        if (off < 0) return fail(CTCB_INVALID_VALUE, "negative logits_row_offsets[%d]", b);
        if (off + t * hp->V > hi) hi = off + t * hp->V;
    }
    *bytes = sizeof(float) * (size_t)hi;
    return CTCB_OK;
}
}

int ctcb_loss_grad_host(const ctcb_problem_t* hp, int device) { return loss_grad_host_impl(hp, device, nullptr); }

int ctcb_loss_grad_host_resident(const ctcb_problem_t* hp, int device, float** dev_grad) {
    if (!dev_grad) return fail(CTCB_INVALID_VALUE, "dev_grad is NULL");
    return loss_grad_host_impl(hp, device, dev_grad);
}

namespace {
// dev_grad != nullptr: the gradient is computed but stays in the device scratch (its address is
// returned); hp->grad is ignored
int loss_grad_host_impl(const ctcb_problem_t* hp, int device, float** dev_grad) {
    if (int rc = validate(hp)) return rc;
    if (device < 0 || device >= 64) return fail(CTCB_INVALID_VALUE, "device %d out of range", device);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device >= ndev)
        return fail(CTCB_UNSUPPORTED, "CUDA device %d not available (there is no CPU path)", device);
    CUDA_TRY(cudaSetDevice(device));
    const int T = hp->T, B = hp->B, V = hp->V, Lmax = hp->Lmax;
    const bool need_grad = hp->grad != nullptr || dev_grad != nullptr;
    // the host entry takes compact buffers only: strides must describe TNC or NTC exactly
    const bool packed = hp->logits_row_offsets != nullptr;
    const bool tnc = !packed && hp->logits_stride_t == (long long)B * V && hp->logits_stride_b == V;
    const bool ntc = packed || (hp->logits_stride_t == V && hp->logits_stride_b == (long long)T * V);
    if (!tnc && !ntc) return fail(CTCB_INVALID_VALUE, "host entry needs compact TNC or NTC logits");
    const long long gst_t = tnc ? (long long)B * V : V, gst_b = tnc ? V : (long long)T * V;      // dense gradient, the logits' layout
    if (need_grad && !dev_grad && (hp->grad_stride_t != gst_t || hp->grad_stride_b != gst_b))
        return fail(CTCB_INVALID_VALUE, "host entry needs a dense grad in the logits' layout");
    if (Lmax > 0 && !((hp->label_stride_b == Lmax && hp->label_stride_l == 1) || (hp->label_stride_b == 1 && hp->label_stride_l == B)))
        return fail(CTCB_INVALID_VALUE, "host entry needs compact NT or TN labels");

    size_t ws_bytes = 0;
    ctcb_workspace_bytes(T, B, V, Lmax, need_grad, &ws_bytes);
    const size_t n_dense = sizeof(float) * (size_t)T * B * V;
    size_t n_log = n_dense;
    if (packed) { if (int rc = packed_logits_bytes(hp, &n_log)) return rc; }
    const size_t n_lab = dt_size(hp->label_dtype) * (size_t)B * (Lmax > 0 ? Lmax : 1);
    const size_t n_dl = hp->data_lengths ? dt_size(hp->data_lengths_dtype) * (size_t)B : 0;
    const size_t n_ll = hp->label_lengths ? dt_size(hp->label_lengths_dtype) * (size_t)B : 0;
    const size_t n_head = hp->head_grad ? sizeof(float) * (size_t)B : 0;
    const size_t n_off = packed ? sizeof(int64_t) * (size_t)B : 0;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o = align_up(o + bytes, 256); return r; };
    const size_t o_ws = take(ws_bytes);
    const size_t o_log = take(n_log), o_grad = take(need_grad ? n_dense : 0), o_lab = take(n_lab),
                 o_dl = take(n_dl), o_ll = take(n_ll), o_head = take(n_head), o_loss = take(sizeof(float) * B),
                 o_sum = take(sizeof(double)), o_stat = take(sizeof(int) * B), o_off = take(n_off);
    std::lock_guard<std::mutex> lk(g_hs_mu);
    HostScratch& hs = g_hs[device];
    if (!hs.stream) {
        if (cudaStreamCreateWithFlags(&hs.stream, cudaStreamNonBlocking) != cudaSuccess)
            return fail(CTCB_MEMOPS_FAILED, "stream creation failed");
    }
    if (hs.bytes < o) {
        if (hs.ptr) cudaFree(hs.ptr);
        hs.ptr = nullptr; hs.bytes = 0;
        if (cudaMalloc(&hs.ptr, o) != cudaSuccess) { cudaGetLastError(); return fail(CTCB_MEMOPS_FAILED, "cudaMalloc(%zu) failed", o); }
        hs.bytes = o;
    }
    char* base = static_cast<char*>(hs.ptr);
    cudaStream_t s = hs.stream;
    if (dev_grad) *dev_grad = reinterpret_cast<float*>(base + o_grad);
#define COPY_TRY(expr) do { if ((expr) != cudaSuccess) return fail(CTCB_MEMOPS_FAILED, "%s: %s", #expr, cudaGetErrorString(cudaGetLastError())); } while (0)
    if (Lmax > 0) COPY_TRY(cudaMemcpyAsync(base + o_lab, hp->labels, n_lab, cudaMemcpyHostToDevice, s));
    if (n_dl) COPY_TRY(cudaMemcpyAsync(base + o_dl, hp->data_lengths, n_dl, cudaMemcpyHostToDevice, s));
    if (n_ll) COPY_TRY(cudaMemcpyAsync(base + o_ll, hp->label_lengths, n_ll, cudaMemcpyHostToDevice, s));
    if (n_head) COPY_TRY(cudaMemcpyAsync(base + o_head, hp->head_grad, n_head, cudaMemcpyHostToDevice, s));
    if (hp->loss_sum) COPY_TRY(cudaMemcpyAsync(base + o_sum, hp->loss_sum, sizeof(double), cudaMemcpyHostToDevice, s));
    if (n_off) COPY_TRY(cudaMemcpyAsync(base + o_off, hp->logits_row_offsets, n_off, cudaMemcpyHostToDevice, s));
    COPY_TRY(cudaMemcpyAsync(base + o_log, hp->logits, n_log, cudaMemcpyHostToDevice, s));
    {
        ctcb_problem_t d = *hp;
        d.logits = reinterpret_cast<float*>(base + o_log);
        d.logits_row_offsets = packed ? reinterpret_cast<const int64_t*>(base + o_off) : nullptr;
        d.grad = need_grad ? reinterpret_cast<float*>(base + o_grad) : nullptr;
        if (dev_grad) { d.grad_stride_t = gst_t; d.grad_stride_b = gst_b; }
        d.labels = base + o_lab;
        d.data_lengths = hp->data_lengths ? base + o_dl : nullptr;
        d.label_lengths = hp->label_lengths ? base + o_ll : nullptr;
        d.head_grad = hp->head_grad ? reinterpret_cast<float*>(base + o_head) : nullptr;
        d.loss = reinterpret_cast<float*>(base + o_loss);
        d.loss_sum = hp->loss_sum ? reinterpret_cast<double*>(base + o_sum) : nullptr;
        d.status = hp->status ? reinterpret_cast<int32_t*>(base + o_stat) : nullptr;
        if (int rc = ctcb_loss_grad(&d, base + o_ws, ws_bytes, s)) return rc;
    }
    COPY_TRY(cudaMemcpyAsync(hp->loss, base + o_loss, sizeof(float) * B, cudaMemcpyDeviceToHost, s));
    if (need_grad && !dev_grad) COPY_TRY(cudaMemcpyAsync(hp->grad, base + o_grad, n_dense, cudaMemcpyDeviceToHost, s));
    if (hp->loss_sum) COPY_TRY(cudaMemcpyAsync(hp->loss_sum, base + o_sum, sizeof(double), cudaMemcpyDeviceToHost, s));
    if (hp->status) COPY_TRY(cudaMemcpyAsync(hp->status, base + o_stat, sizeof(int) * B, cudaMemcpyDeviceToHost, s));
#undef COPY_TRY
    CUDA_TRY(cudaStreamSynchronize(s));
    return CTCB_OK;
}
}  // namespace

// ---- pipelined host entry ---------------------------------------------------------------------
// ctcb_pipe_*: the host entry for a training loop that prefetches.  Batch i+1's inputs cross PCIe on
// a copy stream while batch i's kernels run on the compute stream; the caller collects batch i's loss
// (host) and gradient (device) with ctcb_pipe_wait.  `depth` slots of device buffers rotate; the
// workspace is shared (the compute stream serialises the batches, and one workspace keeps the alpha/beta
// history in L2).
struct ctcb_pipe {
    struct Slot {
        char* in = nullptr; size_t in_bytes = 0;        // input arena (logits, labels, lengths, head)
        char* out = nullptr; size_t out_bytes = 0;      // gradient, loss, loss sum, status
        cudaEvent_t ev_in = nullptr, ev_done = nullptr;
        bool busy = false;
        int64_t ticket = -1;
        float* grad = nullptr;
    };
    int device = 0, depth = 0;
    cudaStream_t s_copy = nullptr, s_comp = nullptr;
    void* ws = nullptr; size_t ws_bytes = 0;
    std::vector<Slot> slots;
    int64_t next = 0;
    int64_t last_h2d = 0;                           // bytes the last submit moved host -> device
    uintptr_t arena_lo = 0, arena_hi = 0;           // a host allocation already verified to hold a whole batch
};

namespace {
// [lo, hi) lies inside ONE allocation known to the driver (page-locked host memory in the unified address
// space): only then may separately described arrays be moved with a single copy over the span between them
// -- the gaps of two unrelated allocations that merely happen to be neighbours could be unmapped or pageable.
bool same_allocation(uintptr_t lo, uintptr_t hi, uintptr_t* range_lo, uintptr_t* range_hi) {
    typedef int (*attr_fn)(void*, int, unsigned long long);
    static attr_fn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuPointerGetAttribute", &f, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<attr_fn>(f);
        cudaGetLastError();
    });
    if (!fn) return false;
    unsigned long long start = 0; size_t size = 0;
    const int kRangeStart = 11, kRangeSize = 12;      // CU_POINTER_ATTRIBUTE_RANGE_START_ADDR / _RANGE_SIZE
    if (fn(&start, kRangeStart, (unsigned long long)lo) != 0 || fn(&size, kRangeSize, (unsigned long long)lo) != 0) return false;
    if (hi > start + size) return false;
    *range_lo = (uintptr_t)start; *range_hi = (uintptr_t)(start + size);
    return true;
}

int pipe_grow(char** ptr, size_t* have, size_t need, cudaStream_t drain) {
    if (*have >= need) return CTCB_OK;
    if (drain) cudaStreamSynchronize(drain);
    if (*ptr) cudaFree(*ptr);
    *ptr = nullptr; *have = 0;
    need = align_up(need + need / 8, 1 << 20);
    if (cudaMalloc(reinterpret_cast<void**>(ptr), need) != cudaSuccess) {
        cudaGetLastError();
        return fail(CTCB_MEMOPS_FAILED, "cudaMalloc(%zu) failed", need);
    }
    *have = need;
    return CTCB_OK;
}
}  // namespace

int ctcb_pipe_create(int device, int depth, ctcb_pipe_t** out) {
    if (!out) return fail(CTCB_INVALID_VALUE, "out is NULL");
    *out = nullptr;
    if (depth < 1 || depth > 8) return fail(CTCB_INVALID_VALUE, "depth %d outside [1,8]", depth);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
        cudaGetLastError();
        return fail(CTCB_UNSUPPORTED, "CUDA device %d not available (there is no CPU path)", device);
    }
    CUDA_TRY(cudaSetDevice(device));
    ctcb_pipe* p = new (std::nothrow) ctcb_pipe();
    if (!p) return fail(CTCB_MEMOPS_FAILED, "out of host memory");
    p->device = device; p->depth = depth;
    p->slots.resize(depth);
    bool ok = cudaStreamCreateWithFlags(&p->s_copy, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&p->s_comp, cudaStreamNonBlocking) == cudaSuccess;
    for (auto& s : p->slots)
        ok = ok && cudaEventCreateWithFlags(&s.ev_in, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&s.ev_done, cudaEventDisableTiming) == cudaSuccess;
    if (!ok) { ctcb_pipe_destroy(p); return fail(CTCB_MEMOPS_FAILED, "stream / event creation failed"); }
    *out = p;
    return CTCB_OK;
}

int ctcb_pipe_destroy(ctcb_pipe_t* p) {
    if (!p) return CTCB_OK;
    cudaSetDevice(p->device);
    if (p->s_comp) cudaStreamSynchronize(p->s_comp);
    if (p->s_copy) cudaStreamSynchronize(p->s_copy);
    for (auto& s : p->slots) {
        if (s.in) cudaFree(s.in);
        if (s.out) cudaFree(s.out);
        if (s.ev_in) cudaEventDestroy(s.ev_in);
        if (s.ev_done) cudaEventDestroy(s.ev_done);
    }
    if (p->ws) cudaFree(p->ws);
    if (p->s_copy) cudaStreamDestroy(p->s_copy);
    if (p->s_comp) cudaStreamDestroy(p->s_comp);
    cudaGetLastError();
    delete p;
    return CTCB_OK;
}

int ctcb_pipe_submit(ctcb_pipe_t* p, const ctcb_problem_t* hp, int64_t* ticket) {
    if (!p || !ticket) return fail(CTCB_INVALID_VALUE, "pipe / ticket is NULL");
    if (int rc = validate(hp)) return rc;
    const int T = hp->T, B = hp->B, V = hp->V, Lmax = hp->Lmax;
    const bool packed = hp->logits_row_offsets != nullptr;
    const bool tnc = !packed && hp->logits_stride_t == (long long)B * V && hp->logits_stride_b == V;
    const bool ntc = packed || (hp->logits_stride_t == V && hp->logits_stride_b == (long long)T * V);
    if (!tnc && !ntc) return fail(CTCB_INVALID_VALUE, "host entry needs compact TNC or NTC logits");
    if (Lmax > 0 && !((hp->label_stride_b == Lmax && hp->label_stride_l == 1) || (hp->label_stride_b == 1 && hp->label_stride_l == B)))
        return fail(CTCB_INVALID_VALUE, "host entry needs compact NT or TN labels");
    const size_t n_dense = sizeof(float) * (size_t)T * B * V;
    size_t n_log = n_dense;
    if (packed) { if (int rc = packed_logits_bytes(hp, &n_log)) return rc; }
    CUDA_TRY(cudaSetDevice(p->device));
    ctcb_pipe::Slot& sl = p->slots[p->next % p->depth];
    if (sl.busy) {   // the caller did not collect this slot's previous batch: its results are overwritten
        CUDA_TRY(cudaEventSynchronize(sl.ev_done));
        sl.busy = false;
    }
    // inputs: {host pointer, bytes}; one copy when they lie in one host arena (batch.py PinnedBatch,
    // the reference's shared-memory collation batchify.py:51), one copy per array otherwise
    struct In { const void* h; size_t n; size_t off; };
    constexpr int NIN = 6;
    In in[NIN] = {
        {hp->logits, n_log, 0},
        {Lmax > 0 ? hp->labels : nullptr, Lmax > 0 ? dt_size(hp->label_dtype) * (size_t)B * Lmax : 0, 0},
        {hp->data_lengths, hp->data_lengths ? dt_size(hp->data_lengths_dtype) * (size_t)B : 0, 0},
        {hp->label_lengths, hp->label_lengths ? dt_size(hp->label_lengths_dtype) * (size_t)B : 0, 0},
        {hp->head_grad, hp->head_grad ? sizeof(float) * (size_t)B : 0, 0},
        {hp->logits_row_offsets, packed ? sizeof(int64_t) * (size_t)B : 0, 0},
    };
    uintptr_t lo = UINTPTR_MAX, hi = 0;
    size_t sum = 0;
    for (const In& a : in)
        if (a.n) {
            const uintptr_t b = reinterpret_cast<uintptr_t>(a.h);
            lo = b < lo ? b : lo; hi = b + a.n > hi ? b + a.n : hi;
            sum += a.n;
        }
    // one copy over the whole span only when the span is one allocation (checked with the driver once per arena)
    bool one_copy = hi - lo <= sum + NIN * 4096;
    if (one_copy && !(lo >= p->arena_lo && hi <= p->arena_hi)) one_copy = same_allocation(lo, hi, &p->arena_lo, &p->arena_hi);
    size_t in_need = 0;
    const size_t skew = lo % 256;            // device addresses congruent to the host's mod 256 (vector loads)
    if (one_copy) {
        for (In& a : in) if (a.n) a.off = skew + (reinterpret_cast<uintptr_t>(a.h) - lo);
        in_need = skew + (hi - lo);
    } else {
        for (In& a : in) if (a.n) { a.off = in_need; in_need = align_up(in_need + a.n, 256); }
    }
    const bool need_grad = true;
    size_t ws_need = 0;
    if (int rc = ctcb_workspace_bytes(T, B, V, Lmax, need_grad, &ws_need)) return rc;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o = align_up(o + bytes, 256); return r; };
    const size_t o_grad = take(n_dense), o_loss = take(sizeof(float) * B), o_sum = take(sizeof(double)),
                 o_stat = take(sizeof(int) * B);
    if (int rc = pipe_grow(&sl.in, &sl.in_bytes, in_need, nullptr)) return rc;
    if (int rc = pipe_grow(&sl.out, &sl.out_bytes, o, nullptr)) return rc;
    if (int rc = pipe_grow(reinterpret_cast<char**>(&p->ws), &p->ws_bytes, ws_need, p->s_comp)) return rc;
#define COPY_TRY(expr) do { if ((expr) != cudaSuccess) return fail(CTCB_MEMOPS_FAILED, "%s: %s", #expr, cudaGetErrorString(cudaGetLastError())); } while (0)
    int64_t moved = 0;
    if (one_copy) {
        COPY_TRY(cudaMemcpyAsync(sl.in + skew, reinterpret_cast<const void*>(lo), hi - lo, cudaMemcpyHostToDevice, p->s_copy));
        moved += (int64_t)(hi - lo);
    } else {
        for (int k = 0; k < NIN; ++k)
            if (in[k].n) { COPY_TRY(cudaMemcpyAsync(sl.in + in[k].off, in[k].h, in[k].n, cudaMemcpyHostToDevice, p->s_copy)); moved += (int64_t)in[k].n; }
    }
    p->last_h2d = moved;
    if (hp->loss_sum) COPY_TRY(cudaMemcpyAsync(sl.out + o_sum, hp->loss_sum, sizeof(double), cudaMemcpyHostToDevice, p->s_copy));
    COPY_TRY(cudaEventRecord(sl.ev_in, p->s_copy));
    COPY_TRY(cudaStreamWaitEvent(p->s_comp, sl.ev_in, 0));
    ctcb_problem_t d = *hp;
    d.logits = reinterpret_cast<const float*>(sl.in + in[0].off);
    d.labels = in[1].n ? sl.in + in[1].off : nullptr;
    d.data_lengths = in[2].n ? sl.in + in[2].off : nullptr;
    d.label_lengths = in[3].n ? sl.in + in[3].off : nullptr;
    d.head_grad = in[4].n ? reinterpret_cast<const float*>(sl.in + in[4].off) : nullptr;
    d.logits_row_offsets = in[5].n ? reinterpret_cast<const int64_t*>(sl.in + in[5].off) : nullptr;
    d.grad = reinterpret_cast<float*>(sl.out + o_grad);
    d.grad_stride_t = tnc ? (long long)B * V : V; d.grad_stride_b = tnc ? V : (long long)T * V;      // dense, the logits' layout
    d.loss = reinterpret_cast<float*>(sl.out + o_loss);
    // A pinned host loss buffer is written by the recursion kernel itself (B stores of 4 bytes over PCIe): a device->host
    // copy of the loss would queue on the copy engine BEHIND the next batch's 2.4 MB host->device copy, the host would see
    // this batch's loss only when that copy is through, and the batch after it would be submitted a copy late (measured:
    // 61 us per cfg2 step with the copy, against 47 us for the host->device copy and 49 us for the kernels alone)
    float* loss_alias = static_cast<float*>(pinned_device_alias(hp->loss));
    if (loss_alias) d.loss = loss_alias;
    d.loss_sum = hp->loss_sum ? reinterpret_cast<double*>(sl.out + o_sum) : nullptr;
    d.status = hp->status ? reinterpret_cast<int32_t*>(sl.out + o_stat) : nullptr;
    if (int rc = ctcb_loss_grad(&d, p->ws, p->ws_bytes, p->s_comp)) return rc;
    if (!loss_alias) COPY_TRY(cudaMemcpyAsync(hp->loss, sl.out + o_loss, sizeof(float) * B, cudaMemcpyDeviceToHost, p->s_comp));
    if (hp->loss_sum) COPY_TRY(cudaMemcpyAsync(hp->loss_sum, sl.out + o_sum, sizeof(double), cudaMemcpyDeviceToHost, p->s_comp));
    if (hp->status) COPY_TRY(cudaMemcpyAsync(hp->status, sl.out + o_stat, sizeof(int) * B, cudaMemcpyDeviceToHost, p->s_comp));
    COPY_TRY(cudaEventRecord(sl.ev_done, p->s_comp));
#undef COPY_TRY
    sl.busy = true;
    sl.ticket = p->next;
    sl.grad = d.grad;
    *ticket = p->next++;
    return CTCB_OK;
}

int ctcb_pipe_last_h2d_bytes(ctcb_pipe_t* p, int64_t* bytes, int32_t* pulled) {
    if (!p) return fail(CTCB_INVALID_VALUE, "pipe is NULL");
    if (bytes) *bytes = p->last_h2d;
    if (pulled) *pulled = 0;        // kept in the signature: the library always copies (DESIGN.md, host entries)
    return CTCB_OK;
}

int ctcb_pipe_wait(ctcb_pipe_t* p, int64_t ticket, float** dev_grad) {
    if (!p) return fail(CTCB_INVALID_VALUE, "pipe is NULL");
    if (ticket < 0 || ticket >= p->next) return fail(CTCB_INVALID_VALUE, "ticket %lld was never issued", (long long)ticket);
    ctcb_pipe::Slot& sl = p->slots[ticket % p->depth];
    if (sl.ticket != ticket)
        return fail(CTCB_INVALID_VALUE, "ticket %lld: its slot was reused by ticket %lld (depth %d)", (long long)ticket,
                    (long long)sl.ticket, p->depth);
    if (sl.busy) {
        CUDA_TRY(cudaEventSynchronize(sl.ev_done));
        sl.busy = false;
    }
    if (dev_grad) *dev_grad = sl.grad;
    return CTCB_OK;
}

int ctcb_scale_rows(float* grad, int64_t stride_t, int64_t stride_b, int32_t T, int32_t B, int32_t V,
                    const float* head_grad, void* stream) {
    if (!grad || !head_grad) return fail(CTCB_INVALID_VALUE, "NULL argument");
    if (T <= 0 || B <= 0 || V <= 0) return fail(CTCB_INVALID_VALUE, "bad shape");
    if (!is_device_ptr(grad) || !is_device_ptr(head_grad)) return fail(CTCB_INVALID_VALUE, "buffers must be CUDA device memory");
    const long long rows = (long long)T * B;
    ctcb::k_scale_rows<<<(unsigned)((rows + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(grad, stride_t, stride_b, T, B, V, head_grad);
    CUDA_TRY(cudaGetLastError());
    g_launches = 1;
    return CTCB_OK;
}

int ctcb_greedy_decode(const float* logits, int64_t stride_t, int64_t stride_b, const void* data_lengths,
                       int32_t data_lengths_dtype, int32_t T, int32_t B, int32_t V, int32_t blank,
                       int32_t* out_tokens, int32_t* out_lengths, void* stream) {
    return ctcb_greedy_decode_unk(logits, stride_t, stride_b, data_lengths, data_lengths_dtype, T, B, V, blank, -1,
                                  out_tokens, out_lengths, stream);
}

int ctcb_greedy_decode_unk(const float* logits, int64_t stride_t, int64_t stride_b, const void* data_lengths,
                           int32_t data_lengths_dtype, int32_t T, int32_t B, int32_t V, int32_t blank, int32_t unk,
                           int32_t* out_tokens, int32_t* out_lengths, void* stream) {
    return ctcb_greedy_decode_typed(logits, CTCB_F32, stride_t, stride_b, data_lengths, data_lengths_dtype, T, B, V, blank, unk,
                                    out_tokens, out_lengths, stream);
}

int ctcb_greedy_decode_typed(const void* logits, int32_t logits_dtype, int64_t stride_t, int64_t stride_b, const void* data_lengths,
                             int32_t data_lengths_dtype, int32_t T, int32_t B, int32_t V, int32_t blank, int32_t unk,
                             int32_t* out_tokens, int32_t* out_lengths, void* stream) {
    if (!logits || !out_tokens || !out_lengths) return fail(CTCB_INVALID_VALUE, "NULL argument");
    if (logits_dtype != CTCB_F32 && logits_dtype != CTCB_BF16)
        return fail(CTCB_INVALID_VALUE, "logits dtype %d is neither CTCB_F32 nor CTCB_BF16 (fp16 logits are not supported)", logits_dtype);
    if (T <= 0 || B <= 0 || V <= 0) return fail(CTCB_INVALID_VALUE, "bad shape");
    if (unk >= V) return fail(CTCB_INVALID_VALUE, "unk %d outside the vocabulary (V=%d; -1 = no <unk> rule)", unk, V);
    if (!is_device_ptr(logits) || !is_device_ptr(out_tokens)) return fail(CTCB_INVALID_VALUE, "buffers must be CUDA device memory");
    const size_t smem = 2 * sizeof(int) * (size_t)T;
    if (smem > 200 * 1024) return fail(CTCB_UNSUPPORTED, "T=%d too long for the decode kernel", T);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (logits_dtype == CTCB_BF16) {
        if (smem > 48 * 1024)
            CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void*>(ctcb::k_greedy_decode<ctcb::bf16>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ctcb::k_greedy_decode<ctcb::bf16><<<B, 256, smem, st>>>(static_cast<const ctcb::bf16*>(logits), stride_t, stride_b, data_lengths,
                                                                data_lengths_dtype, T, B, V, blank, unk < 0 ? -1 : unk, out_tokens, out_lengths);
    } else {
        if (smem > 48 * 1024)
            CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void*>(ctcb::k_greedy_decode<float>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ctcb::k_greedy_decode<float><<<B, 256, smem, st>>>(static_cast<const float*>(logits), stride_t, stride_b, data_lengths,
                                                           data_lengths_dtype, T, B, V, blank, unk < 0 ? -1 : unk, out_tokens, out_lengths);
    }
    CUDA_TRY(cudaGetLastError());
    return CTCB_OK;
}

int ctcb_edit_distance(const int32_t* ref, int64_t ref_stride, const int32_t* ref_len, const int32_t* hyp,
                       int64_t hyp_stride, const int32_t* hyp_len, int32_t B, int32_t max_ref, int32_t max_hyp,
                       int32_t* out_dist, long long* totals, void* stream) {
    if (!ref_len || !hyp_len || !out_dist || (max_ref > 0 && !ref) || (max_hyp > 0 && !hyp))
        return fail(CTCB_INVALID_VALUE, "NULL argument");
    if (B <= 0 || max_ref < 0 || max_hyp < 0) return fail(CTCB_INVALID_VALUE, "bad shape");
    if (!is_device_ptr(ref_len) || !is_device_ptr(hyp_len) || !is_device_ptr(out_dist) || !is_device_ptr(ref) ||
        !is_device_ptr(hyp) || !is_device_ptr(totals))
        return fail(CTCB_INVALID_VALUE, "buffers must be CUDA device memory");
    const size_t smem = sizeof(int) * ((size_t)max_hyp + 2 * ((size_t)max_hyp + 1));
    if (smem > 200 * 1024) return fail(CTCB_UNSUPPORTED, "max_hyp=%d too long for the edit-distance kernel", max_hyp);
    if (smem > 48 * 1024)
        CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void*>(ctcb::k_edit_distance), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ctcb::k_edit_distance<<<B, 128, smem, static_cast<cudaStream_t>(stream)>>>(ref, ref_stride, ref_len, hyp, hyp_stride,
                                                                             hyp_len, max_ref, max_hyp, out_dist, totals);
    CUDA_TRY(cudaGetLastError());
    g_launches = 1;
    return CTCB_OK;
}

// ---- NCCL loss-sum allreduce (dlopen, no link-time dependency) ----------------------------
int ctcb_loss_sum_allreduce(void* nccl_comm, double* dev_values, int32_t count, void* stream) {
    typedef int (*allreduce_fn)(const void*, void*, size_t, int, int, void*, cudaStream_t);
    static allreduce_fn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        const char* names[] = {getenv("CTCB_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
        for (const char* n : names) {
            if (!n) continue;
            if (void* h = dlopen(n, RTLD_NOW | RTLD_GLOBAL)) {
                fn = reinterpret_cast<allreduce_fn>(dlsym(h, "ncclAllReduce"));
                if (fn) break;
            }
        }
    });
    if (!fn) return fail(CTCB_UNSUPPORTED, "ncclAllReduce could not be resolved (set CTCB_NCCL_LIB)");
    if (!nccl_comm || !dev_values || count <= 0) return fail(CTCB_INVALID_VALUE, "bad allreduce arguments");
    const int ncclFloat64 = 8, ncclSum = 0;
    const int rc = fn(dev_values, dev_values, (size_t)count, ncclFloat64, ncclSum, nccl_comm, static_cast<cudaStream_t>(stream));
    if (rc != 0) return fail(CTCB_EXECUTION_FAILED, "ncclAllReduce returned %d", rc);
    return CTCB_OK;
}

// ---- loss-sum exchange over NVLink peer memory ----------------------------------------------
int ctcb_mailbox_create(int device, int rank, int world, int lag, ctcb_mailbox_t** out) {
    if (!out) return fail(CTCB_INVALID_VALUE, "out is NULL");
    *out = nullptr;
    if (world < 1 || world > ctcb::kMailMaxRanks || rank < 0 || rank >= world)
        return fail(CTCB_INVALID_VALUE, "rank %d / world %d outside [0,%d]", rank, world, ctcb::kMailMaxRanks);
    if (lag < 1 || lag > ctcb::kMailMaxLag) return fail(CTCB_INVALID_VALUE, "lag %d outside [1,%d]", lag, ctcb::kMailMaxLag);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
        cudaGetLastError();
        return fail(CTCB_UNSUPPORTED, "CUDA device %d not available (there is no CPU path)", device);
    }
    CUDA_TRY(cudaSetDevice(device));
    ctcb_mailbox* m = new (std::nothrow) ctcb_mailbox();
    if (!m) return fail(CTCB_MEMOPS_FAILED, "out of host memory");
    m->device = device; m->rank = rank; m->world = world;
    const size_t bytes = sizeof(double) * (2 * (size_t)lag * world * ctcb::kMailRow + 8) + sizeof(ctcb::MailboxDev);
    if (cudaMalloc(reinterpret_cast<void**>(&m->local), bytes) != cudaSuccess || cudaMemset(m->local, 0, bytes) != cudaSuccess ||
        cudaDeviceSynchronize() != cudaSuccess) {
        cudaGetLastError();
        if (m->local) cudaFree(m->local);
        delete m;
        return fail(CTCB_MEMOPS_FAILED, "mailbox allocation failed");
    }
    m->dev.rank = rank; m->dev.world = world; m->dev.lag = lag;
    m->dev.counter = reinterpret_cast<unsigned long long*>(m->local + 2 * (size_t)lag * world * ctcb::kMailRow);
    m->dev.peer[rank] = m->local;
    m->dev_d = reinterpret_cast<ctcb::MailboxDev*>(m->local + 2 * (size_t)lag * world * ctcb::kMailRow + 8);
    m->connected = world == 1;
    if (cudaMemcpy(m->dev_d, &m->dev, sizeof(m->dev), cudaMemcpyHostToDevice) != cudaSuccess) {
        cudaGetLastError(); cudaFree(m->local); delete m;
        return fail(CTCB_MEMOPS_FAILED, "mailbox descriptor upload failed");
    }
    *out = m;
    return CTCB_OK;
}

int ctcb_mailbox_handle(ctcb_mailbox_t* m, void* handle64) {
    if (!m || !handle64) return fail(CTCB_INVALID_VALUE, "NULL argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    CUDA_TRY(cudaSetDevice(m->device));
    cudaIpcMemHandle_t h;
    CUDA_TRY(cudaIpcGetMemHandle(&h, m->local));
    memcpy(handle64, &h, 64);
    return CTCB_OK;
}

int ctcb_mailbox_connect(ctcb_mailbox_t* m, const void* handles) {
    if (!m || !handles) return fail(CTCB_INVALID_VALUE, "NULL argument");
    CUDA_TRY(cudaSetDevice(m->device));
    for (int r = 0; r < m->world; ++r) {
        if (r == m->rank || m->opened[r]) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, static_cast<const char*>(handles) + 64 * (size_t)r, 64);
        void* ptr = nullptr;
        const cudaError_t rc = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
        if (rc != cudaSuccess) {
            cudaGetLastError();
            return fail(CTCB_UNSUPPORTED, "cudaIpcOpenMemHandle(rank %d): %s", r, cudaGetErrorString(rc));
        }
        m->opened[r] = ptr;
        m->dev.peer[r] = static_cast<double*>(ptr);
    }
    CUDA_TRY(cudaMemcpy(m->dev_d, &m->dev, sizeof(m->dev), cudaMemcpyHostToDevice));
    m->connected = true;
    return CTCB_OK;
}

static int mailbox_launch(ctcb_mailbox_t* m, double* dev_values, int32_t count, double* dev_out, void* stream, int flush) {
    if (!m || !dev_out || (!flush && !dev_values)) return fail(CTCB_INVALID_VALUE, "NULL argument");
    if (count < 1 || count > ctcb::kMailMaxCount) return fail(CTCB_INVALID_VALUE, "count %d outside [1,%d]", count, ctcb::kMailMaxCount);
    if (!m->connected) return fail(CTCB_INVALID_VALUE, "mailbox is not connected to its peers");
    if (!is_device_ptr(dev_values) || !is_device_ptr(dev_out)) return fail(CTCB_INVALID_VALUE, "buffers must be CUDA device memory");
    ctcb::k_mailbox_exchange<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(m->dev_d, dev_values, count, dev_out, flush);
    CUDA_TRY(cudaGetLastError());
    g_launches = 1;
    return CTCB_OK;
}

int ctcb_mailbox_exchange(ctcb_mailbox_t* m, double* dev_values, int32_t count, double* dev_out, void* stream) {
    return mailbox_launch(m, dev_values, count, dev_out, stream, 0);
}

int ctcb_mailbox_exchange_with_next(ctcb_mailbox_t* m, double* dev_values, int32_t count, double* dev_out) {
    if (!m || !dev_out || !dev_values) return fail(CTCB_INVALID_VALUE, "NULL argument");
    if (count < 1 || count > ctcb::kMailMaxCount) return fail(CTCB_INVALID_VALUE, "count %d outside [1,%d]", count, ctcb::kMailMaxCount);
    if (!m->connected) return fail(CTCB_INVALID_VALUE, "mailbox is not connected to its peers");
    if (!is_device_ptr(dev_values) || !is_device_ptr(dev_out)) return fail(CTCB_INVALID_VALUE, "buffers must be CUDA device memory");
    if (g_xchg.mb) return fail(CTCB_INVALID_VALUE, "an exchange is already waiting for the next gradient launch on this thread");
    g_xchg.mb = m; g_xchg.values = dev_values; g_xchg.out = dev_out; g_xchg.count = count;
    return CTCB_OK;
}

int ctcb_mailbox_flush(ctcb_mailbox_t* m, int32_t count, double* dev_out, void* stream) {
    return mailbox_launch(m, nullptr, count, dev_out, stream, 1);
}

int ctcb_mailbox_destroy(ctcb_mailbox_t* m) {
    if (!m) return CTCB_OK;
    cudaSetDevice(m->device);
    cudaDeviceSynchronize();
    for (int r = 0; r < m->world; ++r) if (m->opened[r]) cudaIpcCloseMemHandle(m->opened[r]);
    if (m->local) cudaFree(m->local);
    cudaGetLastError();
    delete m;
    return CTCB_OK;
}

// ---- DLPack entry ---------------------------------------------------------------------------
namespace {
int dl_dtype(const DLTensor& t, int* out) {
    if (t.dtype.lanes != 1) return 1;
    if (t.dtype.code == kDLInt && t.dtype.bits == 32) { *out = CTCB_I32; return 0; }
    if (t.dtype.code == kDLInt && t.dtype.bits == 64) { *out = CTCB_I64; return 0; }
    if (t.dtype.code == kDLFloat && t.dtype.bits == 32) { *out = CTCB_F32; return 0; }
    if (t.dtype.code == kDLFloat && t.dtype.bits == 64) { *out = CTCB_F64; return 0; }
    return 1;
}
inline void* dl_data(const DLTensor& t) { return static_cast<char*>(t.data) + t.byte_offset; }
inline int64_t dl_stride(const DLTensor& t, int axis) {
    if (t.strides) return t.strides[axis];
    int64_t s = 1;
    for (int i = t.ndim - 1; i > axis; --i) s *= t.shape[i];
    return s;
}
bool dl_cuda(const DLTensor& t) { return t.device.device_type == kDLCUDA || t.device.device_type == kDLCUDAManaged; }
bool dl_vec_ok(const DLManagedTensor* m, int64_t B) {
    if (!m) return true;
    const DLTensor& t = m->dl_tensor;
    return dl_cuda(t) && t.ndim == 1 && t.shape[0] == B && dl_stride(t, 0) == 1;
}
}  // namespace

int ctcb_loss_grad_dlpack(const DLManagedTensor* logits, const DLManagedTensor* labels,
                          const DLManagedTensor* data_lengths, const DLManagedTensor* label_lengths,
                          const DLManagedTensor* head_grad, DLManagedTensor* loss, DLManagedTensor* grad,
                          DLManagedTensor* loss_sum, int32_t blank_last, int32_t layout_flags, void* workspace,
                          size_t workspace_bytes, void* stream) {
    g_launches = 0;
    if (!logits || !labels || !loss) return fail(CTCB_INVALID_VALUE, "logits, labels and loss are required");
    const DLTensor& x = logits->dl_tensor;
    const DLTensor& y = labels->dl_tensor;
    if (!dl_cuda(x) || !dl_cuda(y) || !dl_cuda(loss->dl_tensor))
        return fail(CTCB_INVALID_VALUE, "tensors must live on a CUDA device (there is no CPU path)");
    const bool x_f32 = x.dtype.code == kDLFloat && x.dtype.bits == 32, x_bf16 = x.dtype.code == kDLBfloat && x.dtype.bits == 16;
    if (x.ndim != 3 || !(x_f32 || x_bf16) || x.dtype.lanes != 1)
        return fail(CTCB_INVALID_VALUE, "logits must be a 3-d float32 or bfloat16 tensor");
    const int ldt = x_bf16 ? CTCB_BF16 : CTCB_F32;
    if (dl_stride(x, 2) != 1 && x.shape[2] != 1) return fail(CTCB_INVALID_VALUE, "logits need unit stride on the vocabulary axis");
    if (y.ndim != 2) return fail(CTCB_INVALID_VALUE, "labels must be 2-d");
    const bool ntc = (layout_flags & CTCB_LAYOUT_NTC) != 0, tn = (layout_flags & CTCB_LABEL_TN) != 0;
    ctcb_problem_t p{};
    const int ta = ntc ? 1 : 0, ba = ntc ? 0 : 1;
    p.T = (int32_t)x.shape[ta]; p.B = (int32_t)x.shape[ba]; p.V = (int32_t)x.shape[2];
    p.logits = static_cast<const float*>(dl_data(x));
    p.logits_stride_t = dl_stride(x, ta); p.logits_stride_b = dl_stride(x, ba);
    const int lb = tn ? 1 : 0, ll = tn ? 0 : 1;
    if (y.shape[lb] != p.B) return fail(CTCB_INVALID_VALUE, "labels batch %lld != logits batch %d", (long long)y.shape[lb], p.B);
    p.Lmax = (int32_t)y.shape[ll];
    p.labels = dl_data(y);
    if (dl_dtype(y, &p.label_dtype)) return fail(CTCB_INVALID_VALUE, "labels must be int32/int64/float32/float64");
    p.label_stride_b = dl_stride(y, lb); p.label_stride_l = dl_stride(y, ll);
    p.blank = blank_last ? p.V - 1 : 0;
    p.label_pad = blank_last ? -1 : 0;
    if (!dl_vec_ok(data_lengths, p.B) || !dl_vec_ok(label_lengths, p.B) || !dl_vec_ok(head_grad, p.B) || !dl_vec_ok(loss, p.B))
        return fail(CTCB_INVALID_VALUE, "length/head/loss vectors must be contiguous CUDA (B,) tensors");
    if (data_lengths) {
        p.data_lengths = dl_data(data_lengths->dl_tensor);
        if (dl_dtype(data_lengths->dl_tensor, &p.data_lengths_dtype)) return fail(CTCB_INVALID_VALUE, "bad data_lengths dtype");
    }
    if (label_lengths) {
        p.label_lengths = dl_data(label_lengths->dl_tensor);
        if (dl_dtype(label_lengths->dl_tensor, &p.label_lengths_dtype)) return fail(CTCB_INVALID_VALUE, "bad label_lengths dtype");
    }
    if (head_grad) {
        const DLTensor& h = head_grad->dl_tensor;
        if (h.dtype.code != kDLFloat || h.dtype.bits != 32) return fail(CTCB_INVALID_VALUE, "head_grad must be float32");
        p.head_grad = static_cast<const float*>(dl_data(h));
    }
    {
        const DLTensor& l = loss->dl_tensor;
        if (l.dtype.code != kDLFloat || l.dtype.bits != 32) return fail(CTCB_INVALID_VALUE, "loss must be float32");
        p.loss = static_cast<float*>(dl_data(l));
    }
    if (grad) {
        const DLTensor& g = grad->dl_tensor;
        if (!dl_cuda(g) || g.ndim != 3 || g.dtype.code != x.dtype.code || g.dtype.bits != x.dtype.bits || g.dtype.lanes != 1)
            return fail(CTCB_INVALID_VALUE, "grad must be a 3-d CUDA tensor of the logits' dtype (%s)", x_bf16 ? "bfloat16" : "float32");
        for (int i = 0; i < 3; ++i)
            if (g.shape[i] != x.shape[i]) return fail(CTCB_INVALID_VALUE, "grad shape differs from logits");
        if (dl_stride(g, 2) != 1 && g.shape[2] != 1) return fail(CTCB_INVALID_VALUE, "grad needs unit stride on the vocabulary axis");
        p.grad = static_cast<float*>(dl_data(g));
        p.grad_stride_t = dl_stride(g, ta); p.grad_stride_b = dl_stride(g, ba);
    }
    if (loss_sum) {
        const DLTensor& s = loss_sum->dl_tensor;
        if (!dl_cuda(s) || s.dtype.code != kDLFloat || s.dtype.bits != 64) return fail(CTCB_INVALID_VALUE, "loss_sum must be a float64 CUDA scalar");
        p.loss_sum = static_cast<double*>(dl_data(s));
    }
    const int phase = (layout_flags >> 8) & 3;   // 0: fused, 1: forward (keep history), 2: backward
    if (phase == 1) return enqueue(&p, workspace, workspace_bytes, stream, PH_FORWARD, (layout_flags & CTCB_KEEP_FOR_BACKWARD) != 0, ldt);
    if (phase == 2) return enqueue(&p, workspace, workspace_bytes, stream, PH_BACKWARD, true, ldt);
    return enqueue(&p, workspace, workspace_bytes, stream, p.grad ? (PH_FORWARD | PH_BACKWARD) : PH_FORWARD, p.grad != nullptr, ldt);
}

}  // extern "C"
