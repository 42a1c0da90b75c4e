// ctcb_meet.cuh -- k_meet<P>: the whole CTC training-loss step of one utterance in ONE CTA, for the
// small-vocabulary shapes (V <= 64, L+1 <= 32*P state pairs): rows a3-a9 of SURVEY.md section 8a
// (/root/reference/scripts/swbd/loss.py:134-139, the gluon CTC operator, forward AND backward) in a single
// launch.  Written for the THROUGHPUT regime (BASELINE configs[4]: B = 1024 utterances, sharded over the
// GPUs): the two-kernel path (k_walk + k_grad) sends 8 bytes per lattice state pair, frame and DIRECTION
// through HBM and decodes them again with ~20 integer instructions per state in k_grad; here
//
//   * the alpha walker and the beta walker of an utterance MEET IN THE MIDDLE: each walks its half of the
//     frame blocks storing its history (phase 1), then keeps walking through the OTHER half (phase 2), where
//     every frame's occupancies gamma_t(s) = alpha_t(s) beta'_t(s) / P(l|x) are formed at once from the
//     walker's fresh values and the other walker's stored block.  Only HALF a history crosses the L2 (one
//     direction per frame block, written and read back once by the same SM, last written first read), and
//     the chain is still T steps long, not 2T;
//   * P(l|x) is known at the meeting frame (sum_s alpha_m(s) beta'_m(s)), so the occupancies are normalised
//     by ONE number: a state costs an integer add on the stored high word (the exponent shift
//     2^(offsetA + offsetB - exponent of P)), one DMUL and one conversion -- no per-frame maximum, no
//     mantissa/exponent decode;
//   * one walker warp per direction holds the whole label row (P = 2 or 4 state pairs per lane): no halo,
//     no inter-warp hand-shake inside the recursion.
//
// Warp roles (256 threads): 0 alpha walker, 1 beta walker, 6/7 their emission producers (logits rows ->
// softmax numerators in a shared-memory ring, as k_walk's fused producers), 2,4 the alpha side's helpers,
// 3,5 the beta side's (one helper on each of the SM's four sub-partitions).  A walker hands every finished frame block (8 frames of high words + the block's
// exponent offsets, 9 rows) to its side's helpers through a 2-deep shared-memory ring; helper h takes the
// blocks of parity h.  Phase 1: the helper sends the block to the workspace with one bulk store
// (cp.async.bulk.global.shared::cta).  Phase 2: it fetches the other direction's block of the same frames
// with one bulk load, forms the occupancies, sums them per label in rank order (deterministic, no
// atomics), and writes grad = head * (softmax - occupancy) rows, coalesced, in the caller's layout.
// Number format, renormalisation and the emission floor are k_walk's (ctcb_kernels.cuh, DESIGN.md 4).
#pragma once
#include "ctcb_kernels.cuh"

namespace ctcb {

#ifndef MEET_UNROLL
#define MEET_UNROLL 2
#endif
constexpr int kMeetUnroll = MEET_UNROLL;   // walker steps unrolled per loop trip
constexpr int kMeetES = 2;            // emission ring depth per direction (frame blocks)
constexpr int kMeetFR = 8;            // ring of per-frame {row max, log2 sum} blocks (producer -> helpers)
constexpr int kHR = kG + 1;           // rows of a history block: kG frames + the block's exponent offsets
constexpr unsigned kMeetSpinIters = 1u << 24;   // try_wait rounds any wait inside the CTA may take before the kernel traps

struct MeetArgs {
    Problem p;
    int2* hist;            // (B, NB, kHR, 32*P) history blocks; block n is written by ONE direction (alpha: n < NA_b)
    int NB;
    long long* trace;      // debug only (scripts/ubench/meet_trace.cu); nullptr in the product
};

#ifdef CTCB_TRACE
#define MEET_TP(n_, id_) do { if (c.trace && c.b == 0 && (threadIdx.x & 31) == 0 && (n_) < 256) \
    c.trace[((size_t)(threadIdx.x >> 5) * 256 + (size_t)(n_)) * 8 + (id_)] = clock64(); } while (0)
#else
#define MEET_TP(n_, id_) do { } while (0)
#endif

struct MeetSmem {          // byte offsets into the dynamic shared memory
    uint32_t ering[2], hring[2], oring[2], rowbuf, zsum, lab, rank, runv, frr[2], juncv, junce, lzp, pinfo, bars, total;
};
constexpr int kMeetBars = 2 * kMeetES * 2 + 2 * 2 * 2 + 2 * 2 + 2 + 2;   // fullE, emptyE, fullH, emptyH, fullO, J, J2, HD[2]

__host__ __device__ inline MeetSmem meet_smem_layout(int P, int V, int Lp) {
    MeetSmem m;
    const uint32_t PW = 32u * P, stageE = (uint32_t)V * kEC * 8u, blockH = (uint32_t)kHR * PW * 8u;
    uint32_t o = 0;
    auto take = [&](uint32_t bytes) { uint32_t r = o; o = (o + bytes + 127u) & ~127u; return r; };
    for (int d = 0; d < 2; ++d) m.ering[d] = take(kMeetES * stageE);
    for (int d = 0; d < 2; ++d) m.hring[d] = take(2 * blockH);
    for (int d = 0; d < 2; ++d) m.oring[d] = take(2 * blockH);
    m.rowbuf = take(4 * 4 * PW * 4);
    m.zsum = take(4 * kG * 4);
    m.lab = take((uint32_t)Lp * 4 + 16);
    m.rank = take((uint32_t)PW * 4);
    m.runv = take(64 * 8);
    for (int d = 0; d < 2; ++d) m.frr[d] = take(kMeetFR * kG * 8);
    m.juncv = m.rowbuf;                  // the meeting record is dead before the first helper touches its row buffer
    m.junce = m.rowbuf + PW * 16;
    m.lzp = take(2 * 8 * 8);
    m.pinfo = take(16);
    m.bars = take(kMeetBars * 8);
    m.total = o;
    return m;
}

struct MeetCtx {
    int b, Tb, Lb, NQ, rlast, NA, V, blank;
    unsigned char* smem;
    uint32_t base;          // shared-window address of smem
    MeetSmem m;
    uint64_t* bars;
    long long* trace;
    __device__ __forceinline__ uint64_t* fullE(int d, int s) const { return bars + d * kMeetES + s; }
    __device__ __forceinline__ uint64_t* emptyE(int d, int s) const { return bars + 2 * kMeetES + d * kMeetES + s; }
    __device__ __forceinline__ uint64_t* fullH(int d, int s) const { return bars + 4 * kMeetES + d * 2 + s; }
    __device__ __forceinline__ uint64_t* emptyH(int d, int s) const { return bars + 4 * kMeetES + 4 + d * 2 + s; }
    __device__ __forceinline__ uint64_t* fullO(int d, int s) const { return bars + 4 * kMeetES + 8 + d * 2 + s; }
    __device__ __forceinline__ uint64_t* J() const { return bars + 4 * kMeetES + 12; }
    __device__ __forceinline__ uint64_t* J2() const { return bars + 4 * kMeetES + 13; }
    __device__ __forceinline__ uint64_t* HD(int d) const { return bars + 4 * kMeetES + 14 + d; }
    __device__ __forceinline__ int n1(int d) const { return d ? NQ - NA : NA; }      // phase-1 blocks of direction d
};

// bounded wait: a protocol error inside the CTA ends the kernel with a trap (an error the host sees), not a hang
__device__ __forceinline__ bool mbar_try(uint64_t* bar, uint32_t parity) {      // try_wait: the hardware suspends the thread for a while
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait_b(uint64_t* bar, uint32_t parity) {
    // try_wait suspends the thread in hardware for a while; the iteration cap (seconds) turns a protocol error into a trap
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .u32 k;\n\t"
        "mov.u32 k, 0;\n\t"
        "W_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra D_%=;\n\t"
        "add.u32 k, k, 1;\n\t"
        "setp.lt.u32 p, k, %2;\n\t"
        "@p bra W_%=;\n\t"
        "trap;\n\t"
        "D_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity), "r"(kMeetSpinIters) : "memory");
}
__device__ __forceinline__ void mbar_wait_sleep(uint64_t* bar, uint32_t parity) { mbar_wait_b(bar, parity); }
__device__ __forceinline__ void sts_v4(uint32_t addr, int4 v) {
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void sts_v2(uint32_t addr, int2 v) {
    asm volatile("st.shared.v2.b32 [%0], {%1,%2};" ::"r"(addr), "r"(v.x), "r"(v.y) : "memory");
}
__device__ __forceinline__ int2 lds_v2(uint32_t addr) {
    int2 v; asm volatile("ld.shared.v2.b32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr) : "memory"); return v;
}
__device__ __forceinline__ int lds_s32(uint32_t addr) {
    int v; asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory"); return v;
}
__device__ __forceinline__ float lds_f32(uint32_t addr) {
    float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory"); return v;
}
__device__ __forceinline__ void sts_f32(uint32_t addr, float v) {
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ double warp_sum_f64(double s) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        s += __hiloint2double(__shfl_xor_sync(0xffffffffu, __double2hiint(s), o), __shfl_xor_sync(0xffffffffu, __double2loint(s), o));
    return s;
}

// ---------------------------------------------------------------------------------------------------------
// walker warp of direction DIR: all NQ frame blocks of the utterance in its walking order; every block's
// history goes to the direction's shared-memory ring.  At walking index n1(DIR) -- the meeting point -- the
// alpha walker publishes its state, the beta walker forms P(l|x), the loss and the occupancies' scale.
// ---------------------------------------------------------------------------------------------------------
template <int P>
__device__ __forceinline__ void meet_walker(const MeetCtx& c, const Problem& p, const int DIR) {
    constexpr int PW = 32 * P;
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int Lb = c.Lb, NQ = c.NQ;
    const int g0 = lane * P;
    const uint32_t stageE = (uint32_t)c.V * kEC * 8u, blockH = (uint32_t)kHR * PW * 8u;
    const uint32_t ering = c.base + c.m.ering[DIR], hring = c.base + c.m.hring[DIR];
    const int* lab = reinterpret_cast<const int*>(c.smem + c.m.lab);
    const uint32_t bcol = (uint32_t)c.blank * (kEC * 8u);
    bool skip[P]; uint32_t ccol[P];
#pragma unroll
    for (int q = 0; q < P; ++q) {
        const int g = g0 + q;
        const bool vl = g < Lb;
        const int cur = vl ? (DIR ? lab[Lb - 1 - g] : lab[g]) : -1;
        const int prv = (vl && g >= 1) ? (DIR ? lab[Lb - g] : lab[g - 1]) : -2;
        skip[q] = vl && g >= 1 && cur != prv;
        ccol[q] = vl ? (uint32_t)cur * (kEC * 8u) : bcol;
    }
    double bm[P], lm[P], fb[P], fls[P], flb[P]; int eb[P], el[P];
#pragma unroll
    for (int q = 0; q < P; ++q) {
        bm[q] = 0.0; lm[q] = 0.0; eb[q] = 0; el[q] = 0;
        fb[q] = 1.0; flb[q] = 1.0; fls[q] = skip[q] ? 1.0 : 0.0;
    }
    if (lane == 0) bm[0] = 1.0;                 // virtual state before the first frame = delta(s = 0)
    double pm = 0.0;                            // the left neighbour's label state for the coming step
    const int N1 = c.n1(DIR);

    auto meeting_point = [&]() {
            // ---- the meeting point ----
            if (DIR == 0) {
                // alpha_m (emission applied), full fp64, and its offsets: read by the beta walker
#pragma unroll
                for (int q = 0; q < P; ++q) {
                    double* jv = reinterpret_cast<double*>(c.smem + c.m.juncv) + 2 * (g0 + q);
                    jv[0] = bm[q]; jv[1] = lm[q];
                    reinterpret_cast<int2*>(c.smem + c.m.junce)[g0 + q] = make_int2(eb[q], el[q]);
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(c.J());
            } else {
                mbar_wait_b(c.J(), 0);
                // beta'_m: the sums of the coming step, before its emission.  P(l|x) = sum_s alpha_m(s) beta'_m(s)
                const double* jv = reinterpret_cast<const double*>(c.smem + c.m.juncv);
                const int2* je = reinterpret_cast<const int2*>(c.smem + c.m.junce);
                double ma[2 * P], mb[2 * P]; int ex[2 * P];
                int emax = 2 * kZeroE;
#pragma unroll
                for (int q = 0; q < P; ++q) {
                    const int g = g0 + q;
                    const double prev = q == 0 ? pm : lm[q - 1];
                    const double sb = fma(prev, fb[q], bm[q]);
                    const double sl = fma(prev, fls[q], fma(bm[q], flb[q], lm[q]));
                    const int ib = max(Lb - g, 0), il = max(Lb - 1 - g, 0);
                    const double ab = jv[2 * ib], al = jv[2 * il + 1];
                    const int eab = je[ib].x, eal = je[il].y;
                    const bool vb = g <= Lb && sb > 0.0 && ab > 0.0, vl = g < Lb && sl > 0.0 && al > 0.0;
                    ma[2 * q] = vb ? dmant(ab) : 0.0; mb[2 * q] = vb ? dmant(sb) : 0.0;
                    ex[2 * q] = vb ? eb[q] + eab + dexp(sb) + dexp(ab) : 2 * kZeroE;
                    ma[2 * q + 1] = vl ? dmant(al) : 0.0; mb[2 * q + 1] = vl ? dmant(sl) : 0.0;
                    ex[2 * q + 1] = vl ? el[q] + eal + dexp(sl) + dexp(al) : 2 * kZeroE;
                    emax = max(emax, max(ex[2 * q], ex[2 * q + 1]));
                }
                emax = __reduce_max_sync(FULL, emax);
                double s = 0.0;
#pragma unroll
                for (int k = 0; k < 2 * P; ++k) s += ma[k] * mb[k] * pow2c(max(ex[k] - emax, -2000));
                s = warp_sum_f64(s);
                // s in [1, 4 * pairs): P(l|x) = s * 2^emax.  (A feasible utterance has s > 0.)
                const int EP = emax + dexp(s);
                const double mP = dmant(s);
                if (lane == 0) {
                    int* pi = reinterpret_cast<int*>(c.smem + c.m.pinfo);
                    pi[0] = EP;
                    reinterpret_cast<float*>(pi)[1] = (float)(1.0 / mP);
                    double lz = 0.0;
                    const double* lzp = reinterpret_cast<const double*>(c.smem + c.m.lzp);
#pragma unroll
                    for (int k = 0; k < 2; ++k) lz += lzp[k];
                    const double nll = -kLn2 * ((double)EP + log2(mP) - lz);
                    p.loss[c.b] = (float)nll;
                    if (p.loss_sum) atomicAdd(p.loss_sum, nll);
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(c.J2());
            }
    };
    int n = 0;
#pragma unroll 1
    for (int phase = 0; phase < 2; ++phase) {
    const int n_end = phase ? NQ : N1;
#pragma unroll 1
    for (; n < n_end; ++n) {
        const int blk = DIR ? NQ - 1 - n : n;
        const int ns = blk == NQ - 1 ? c.rlast : kG;
        const int se = n % kMeetES, ke = n / kMeetES, sh = n & 1, kh = n >> 1;
        const uint32_t stage_base = ering + (uint32_t)se * stageE;
        const uint32_t hstage = hring + (uint32_t)sh * blockH;
        MEET_TP(n, 0);
        mbar_wait_b(c.fullE(DIR, se), (uint32_t)(ke & 1));
        MEET_TP(n, 1);
        const int j0 = DIR ? ns - 1 : 0;
        double yb, yl[P];
        yb = lds_f64(stage_base + bcol + (uint32_t)j0 * 8u);
#pragma unroll
        for (int q = 0; q < P; ++q) yl[q] = lds_f64(stage_base + ccol[q] + (uint32_t)j0 * 8u);
        // renormalise?  (some state drifted past 2^+-kDrift)
        int bad = 0;
        {
            constexpr unsigned LO = (1023u - kDrift) << 20, SPAN = (2u * kDrift + 1u) << 20;
#pragma unroll
            for (int q = 0; q < P; ++q) {
                const unsigned hb = (unsigned)__double2hiint(bm[q]), hl = (unsigned)__double2hiint(lm[q]);
                bad |= (int)(hb != 0u) & (int)(hb - LO >= SPAN);
                bad |= (int)(hl != 0u) & (int)(hl - LO >= SPAN);
            }
        }
        if (__builtin_expect(__any_sync(FULL, bad != 0), 0)) {
            int natb[P], natl[P], am[P];
            bool hard = false;
#pragma unroll
            for (int q = 0; q < P; ++q) {
                natb[q] = bm[q] != 0.0 ? eb[q] + dexp(bm[q]) : kZeroE;
                natl[q] = lm[q] != 0.0 ? el[q] + dexp(lm[q]) : kZeroE;
                am[q] = max(natb[q], natl[q]);
                hard |= bm[q] == 0.0 || lm[q] == 0.0 || natb[q] - kD > natl[q];
            }
            {
                int pa = __shfl_up_sync(FULL, am[P - 1], 1);
                if (lane == 0) pa = kZeroE;
#pragma unroll
                for (int q = 0; q < P; ++q) { hard |= pa - kD > min(natb[q], natl[q]); pa = am[q]; }
            }
            if (__any_sync(FULL, hard)) {
                // R(g) = max(a(g), R(g-1) - kD): in the lane, then across lanes (decay P*kD per lane)
                int x = am[0], anymax = am[0];
#pragma unroll
                for (int q = 1; q < P; ++q) { x = max(am[q], x - kD); anymax = max(anymax, am[q]); }
#pragma unroll
                for (int i = 1; i < 32; i <<= 1) {
                    const int y = __shfl_up_sync(FULL, x, i);
                    if (lane >= i) x = max(x, y - i * P * kD);
                }
                x = max(x, 2 * kZeroE);
                int Rp = __shfl_up_sync(FULL, x, 1);
                if (lane == 0) Rp = kZeroE;
                const unsigned nz = __ballot_sync(FULL, anymax > kZeroE);
                const int fl = nz ? 31 - __clz(nz) : -1;            // lane of the wavefront's last nonzero pair
                int F = 0;
                if (nz) F = __shfl_sync(FULL, x, fl);
                const bool beyond = lane > fl;                      // exactly-zero states beyond the front take F
#pragma unroll
                for (int q = 0; q < P; ++q) {
                    const int base = Rp - kD;
                    const int zoff = beyond ? F : base;
                    const int neb = natb[q] > kZeroE ? max(natb[q], base) : zoff;
                    const int nel = natl[q] > kZeroE ? max(natl[q], max(natb[q] - kD, base)) : (natb[q] > kZeroE ? neb : zoff);
                    bm[q] *= pow2c(eb[q] - neb);
                    lm[q] *= pow2c(el[q] - nel);
                    eb[q] = neb; el[q] = nel;
                    Rp = max(max(am[q], Rp - kD), 2 * kZeroE);
                }
            } else {
#pragma unroll
                for (int q = 0; q < P; ++q) {
                    bm[q] = dmant(bm[q]); lm[q] = dmant(lm[q]);
                    eb[q] = natb[q]; el[q] = natl[q];
                }
            }
            {                                                   // values moved: refresh the pre-shuffled neighbour
                const double q = shfl_up_f64(lm[P - 1]);
                pm = lane != 0 ? q : 0.0;
            }
            int ep = __shfl_up_sync(FULL, el[P - 1], 1);
            if (lane == 0) ep = eb[0];
#pragma unroll
            for (int q = 0; q < P; ++q) {
                fb[q] = pow2c(ep - eb[q]);
                fls[q] = skip[q] ? pow2c(ep - el[q]) : 0.0;
                flb[q] = pow2c(eb[q] - el[q]);
                ep = el[q];
            }
        }
        // the ring slot of this block's history: free once its helper is done with block n - 2
        MEET_TP(n, 2);
        if (kh > 0) mbar_wait_b(c.emptyH(DIR, sh), (uint32_t)((kh - 1) & 1));
        MEET_TP(n, 3);
        {
            const uint32_t orow = hstage + (uint32_t)(kG * PW + g0) * 8u;
            if (P % 2 == 0) {
#pragma unroll
                for (int q = 0; q < P; q += 2) sts_v4(orow + q * 8u, make_int4(eb[q], el[q], eb[(q + 1) % P], el[(q + 1) % P]));
            } else {
#pragma unroll
                for (int q = 0; q < P; ++q) sts_v2(orow + q * 8u, make_int2(eb[q], el[q]));
            }
        }
        auto step = [&](int j, int nj) {
            double nyb = 0.0, nyl[P];
            if (nj >= 0) {
                nyb = lds_f64(stage_base + bcol + (uint32_t)nj * 8u);
#pragma unroll
                for (int q = 0; q < P; ++q) nyl[q] = lds_f64(stage_base + ccol[q] + (uint32_t)nj * 8u);
            }
            double t0[P], sb[P], sl[P];
#pragma unroll
            for (int q = P - 1; q >= 0; --q) {
                const double prev = q == 0 ? pm : lm[q - 1];
                t0[q] = fma(bm[q], flb[q], lm[q]);
                sb[q] = fma(prev, fb[q], bm[q]);
            }
#pragma unroll
            for (int q = P - 1; q >= 0; --q) {
                const double prev = q == 0 ? pm : lm[q - 1];
                sl[q] = fma(prev, fls[q], t0[q]);
            }
#pragma unroll
            for (int q = P - 1; q >= 0; --q) lm[q] = sl[q] * yl[q];
            const double pm_next = shfl_up_f64(lm[P - 1]);
#pragma unroll
            for (int q = P - 1; q >= 0; --q) bm[q] = sb[q] * yb;
            {
                int2 hw[P];
#pragma unroll
                for (int q = 0; q < P; ++q)
                    hw[q] = DIR ? make_int2(__double2hiint(sb[q]), __double2hiint(sl[q]))
                                : make_int2(__double2hiint(bm[q]), __double2hiint(lm[q]));
                const uint32_t dst = hstage + (uint32_t)(j * PW + g0) * 8u;
                if (P % 2 == 0) {
#pragma unroll
                    for (int q = 0; q < P; q += 2) sts_v4(dst + q * 8u, make_int4(hw[q].x, hw[q].y, hw[(q + 1) % P].x, hw[(q + 1) % P].y));
                } else {
#pragma unroll
                    for (int q = 0; q < P; ++q) sts_v2(dst + q * 8u, hw[q]);
                }
            }
            pm = lane != 0 ? pm_next : 0.0;
            if (nj >= 0) {
                yb = nyb;
#pragma unroll
                for (int q = 0; q < P; ++q) yl[q] = nyl[q];
            }
        };
        // one rolled step loop for full and partial blocks: the CTA's eight warps run five different loops, and
        // together they have to stay inside the SM's instruction cache
#pragma unroll kMeetUnroll
        for (int jj = 0; jj < ns; ++jj) {
            const int j = DIR ? ns - 1 - jj : jj;
            const int nj = jj + 1 < ns ? (DIR ? j - 1 : j + 1) : -1;
            step(j, nj);
        }
        MEET_TP(n, 4);
        __syncwarp();
        if (lane == 0) { mbar_arrive(c.fullH(DIR, sh)); mbar_arrive(c.emptyE(DIR, se)); }
        MEET_TP(n, 5);
    }
    if (phase == 0) meeting_point();
    }
}

// ---------------------------------------------------------------------------------------------------------
// producer warp of direction DIR: logits rows -> emission blocks (softmax numerators, fp64, frame-minor) in the
// direction's ring, in the walker's order; {row max, log2 sum} of every frame for the helpers' softmax; the
// sum of log2 sums over the direction's phase-1 frames for the loss.  A lane owns the symbols v = lane and
// lane + 32 (coalesced row reads); four frames per loop trip, the next four frames' rows in flight meanwhile.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void meet_producer(const MeetCtx& c, const Problem& p, const int DIR) {
    constexpr unsigned FULL = 0xffffffffu;
    constexpr int CPL = 16;                                        // symbols per lane, at most (V <= 64)
    const int lane = threadIdx.x & 31, V = c.V, NQ = c.NQ, Tb = c.Tb;
    const int fj = lane >> 2, s4 = lane & 3;                       // frame of the block; this lane's symbols: s4, s4 + 4, ...
    const float* base = utt_logits(p, c.b);
    const float kMinProb = 7.888609052210118e-31f;                 // 2^kMinLog2
    const uint32_t stageE = (uint32_t)V * kEC * 8u;
    const uint32_t ering = c.base + c.m.ering[DIR];
    float2* frr = reinterpret_cast<float2*>(c.smem + c.m.frr[DIR]);
    const int N1 = c.n1(DIR);
    float x[CPL];
    auto load_blk = [&](int n) {
        const int t = (DIR ? NQ - 1 - n : n) * kG + fj;
        const float* row = base + (long long)t * p.st_t + s4;
        const bool valid = n < NQ && t < Tb;
#pragma unroll
        for (int i = 0; i < CPL; ++i) x[i] = (valid && s4 + 4 * i < V) ? __ldg(row + 4 * i) : -INFINITY;
    };
    // rows of the block three ahead -> L2 (one 128-byte line per lane and request: 8 rows of V <= 64 floats)
    auto prefetch_blk = [&](int n) {
        if (n >= NQ) return;
        const int t = (DIR ? NQ - 1 - n : n) * kG + fj;
        const float* row = base + (long long)t * p.st_t + s4 * 32;
        if (t < Tb && s4 * 32 < V) asm volatile("prefetch.global.L2 [%0];" ::"l"(row));
    };
    double ls = 0.0;
    bool floored = false;
    prefetch_blk(1); prefetch_blk(2);
    load_blk(0);
#pragma unroll 1
    for (int n = 0; n < NQ; ++n) {
        MEET_TP(n, 0);
        prefetch_blk(n + 3);
        const int blk = DIR ? NQ - 1 - n : n;
        const bool valid = blk * kG + fj < Tb;
        float mx = x[0];
#pragma unroll
        for (int i = 1; i < CPL; ++i) mx = fmaxf(mx, x[i]);
        mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, 1));
        mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, 2));
        const int st = n % kMeetES, use = n / kMeetES;
        MEET_TP(n, 1);
        if (use > 0) mbar_wait_sleep(c.emptyE(DIR, st), (uint32_t)((use - 1) & 1));
        MEET_TP(n, 2);
        const uint32_t dst = ering + (uint32_t)st * stageE + (uint32_t)s4 * (kEC * 8u) + (uint32_t)fj * 8u;
        float sm = 0.0f;
#pragma unroll
        for (int i = 0; i < CPL; ++i) {
            const bool on = s4 + 4 * i < V;
            const float e = (valid && on) ? fast_ex2((x[i] - mx) * kLog2e) : 0.0f;
            sm += e;
            floored |= valid && on && e < kMinProb;
            if (on) sts_f64(dst + (uint32_t)(4 * i) * (kEC * 8u), valid ? (double)fmaxf(e, kMinProb) : 0.0);
        }
        sm += __shfl_xor_sync(FULL, sm, 1);
        sm += __shfl_xor_sync(FULL, sm, 2);
        const float l2 = valid ? log2f(sm) : 0.0f;
        // sum over the block's frames in frame order (lane 4*j holds frame j's): fixed order for the loss
        float lsum = 0.0f;
#pragma unroll
        for (int j = 0; j < kG; ++j) lsum += __shfl_sync(FULL, l2, 4 * j);
        if (n < N1) ls += (double)lsum;
        if (s4 == 0) frr[(blk % kMeetFR) * kG + fj] = make_float2(mx, l2);
        if (lane == 0 && n < N1) reinterpret_cast<double*>(c.smem + c.m.lzp)[DIR] = ls;   // before the arrive: the walker's acquire covers it
        __syncwarp();
        if (lane == 0) mbar_arrive(c.fullE(DIR, st));
        MEET_TP(n, 3);
        load_blk(n + 1);                       // into the same registers: lands while this warp waits for the ring slot
    }
    if (DIR == 0 && p.status && __any_sync(FULL, floored) && lane == 0) atomicOr(p.status + c.b, UTT_WIDE_LOGITS);
}

// ---------------------------------------------------------------------------------------------------------
// helper warp h of side SIDE: the side's frame blocks of walking-order parity h.
// ---------------------------------------------------------------------------------------------------------
template <int P>
__device__ __forceinline__ void meet_helper(const MeetCtx& c, const Problem& p, int2* hist_b, const int SIDE, const int h) {
    constexpr int PW = 32 * P;
    constexpr unsigned FULL = 0xffffffffu;
    constexpr uint32_t blockH = (uint32_t)kHR * PW * 8u;
    const int lane = threadIdx.x & 31;
    const int Lb = c.Lb, NQ = c.NQ, Tb = c.Tb, V = c.V;
    const int N1 = c.n1(SIDE);
    const uint32_t hstage = c.base + c.m.hring[SIDE] + (uint32_t)h * blockH;
    const uint32_t ostage = c.base + c.m.oring[SIDE] + (uint32_t)h * blockH;
    unsigned char* ostage_p = c.smem + c.m.oring[SIDE] + (size_t)h * blockH;
    unsigned char* hstage_p = c.smem + c.m.hring[SIDE] + (size_t)h * blockH;
    float* grad_b = p.grad + c.b * p.gst_b;

    // rows past the utterance's length: exact zeros (the four helpers of the CTA share them)
    for (int t = Tb + SIDE * 2 + h; t < p.T; t += 4) {
        float* grow = grad_b + (long long)t * p.gst_t;
        for (int v = lane; v < V; v += 32) grow[v] = 0.0f;
    }

    int n = h, u = 0;                     // walking index of this helper's next block; its use count of the ring slot
    // ---- phase 1: the walker's blocks go to the workspace, one bulk store each ----
#pragma unroll 1
    for (; n < N1; n += 2, ++u) {
        const int blk = SIDE ? NQ - 1 - n : n;
        MEET_TP(n, 0);
        mbar_wait_sleep(c.fullH(SIDE, h), (uint32_t)(u & 1));
        MEET_TP(n, 1);
        if (lane == 0) {
            tma_store_1d(hist_b + (size_t)blk * kHR * PW, hstage_p, blockH);
            tma_store_wait_read();
            mbar_arrive(c.emptyH(SIDE, h));
        }
        __syncwarp();
        MEET_TP(n, 2);
    }
    if (lane == 0) {
        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");      // this helper's blocks are in global memory
        mbar_arrive(c.HD(SIDE));
    }
    __syncwarp();
    if (n >= NQ) return;
    // ---- phase 2 ----
    mbar_wait_sleep(c.HD(1 - SIDE), 0);          // the other direction's blocks are in global memory
    mbar_wait_sleep(c.J2(), 0);                  // P(l|x) is known
    const int EP = *reinterpret_cast<const int*>(c.smem + c.m.pinfo);
    const float rP = reinterpret_cast<const float*>(c.smem + c.m.pinfo)[1];
    const float head = p.head ? p.head[c.b] : 1.0f;
    auto fetch = [&](int nn) {                   // the other direction's block of walking index nn -> this helper's slot
        const int blk = SIDE ? NQ - 1 - nn : nn;
        mbar_expect_tx(c.fullO(SIDE, h), blockH);
        tma_load_1d(ostage_p, hist_b + (size_t)blk * kHR * PW, blockH, c.fullO(SIDE, h));
    };
    if (lane == 0) fetch(n);
    // A = the alpha walker's block (pair coordinates g), B = the beta walker's (reversed slots)
    const uint32_t Abase = SIDE == 0 ? hstage : ostage, Bbase = SIDE == 0 ? ostage : hstage;
    const int* rank = reinterpret_cast<const int*>(c.smem + c.m.rank);
    const int2* runv = reinterpret_cast<const int2*>(c.smem + c.m.runv);
    // per helper: two frames of label occupancies in rank order, then their inclusive prefix sums
    const uint32_t rowbuf = c.base + c.m.rowbuf + (uint32_t)(SIDE * 2 + h) * (4 * PW) * 4u;    // [2 frames][PW] gamma, [2 frames][PW] prefix sums
    const uint32_t sumbuf = rowbuf + 2u * PW * 4u;
    const float2* frr = reinterpret_cast<const float2*>(c.smem + c.m.frr[SIDE]);
    int ibb[P], ibl[P], rk[P];
#pragma unroll
    for (int q = 0; q < P; ++q) {
        const int g = q * 32 + lane;
        ibb[q] = max(Lb - g, 0); ibl[q] = max(Lb - 1 - g, 0);
        rk[q] = g < Lb ? rank[g] : g;
    }
    const int v0 = lane, v1 = lane + 32;
    const bool has0 = v0 < V, has1 = v1 < V;
    // the run [start, end) of each of this lane's two symbols in rank order -> prefix-sum slots end-1 and start-1
    const int2 run0 = has0 ? runv[v0] : make_int2(0, 0), run1 = has1 ? runv[v1] : make_int2(0, 0);
    const float* xbase = utt_logits(p, c.b);
    int uo = 0;
#pragma unroll 1
    for (; n < NQ; n += 2, ++u, ++uo) {
        const int blk = SIDE ? NQ - 1 - n : n;
        const int ns = blk == NQ - 1 ? c.rlast : kG;
        const int t0 = blk * kG;
        // the first two frames' logits (each loop trip loads the next trip's)
        float xa[2], xb[2];
#pragma unroll
        for (int f = 0; f < 2; ++f) {
            const float* row = xbase + (long long)(t0 + f) * p.st_t;
            xa[f] = (f < ns && has0) ? __ldg(row + v0) : 0.0f;
            xb[f] = (f < ns && has1) ? __ldg(row + v1) : 0.0f;
        }
        MEET_TP(n, 0);
        mbar_wait_sleep(c.fullO(SIDE, h), (uint32_t)(uo & 1));
        MEET_TP(n, 1);
        mbar_wait_sleep(c.fullH(SIDE, h), (uint32_t)(u & 1));
        MEET_TP(n, 2);
        // exponent shift of every state of the block: offsets of both directions minus the exponent of P(l|x)
        int dsb[P], dsl[P];
#pragma unroll
        for (int q = 0; q < P; ++q) {
            const int g = q * 32 + lane;
            const int2 oa = lds_v2(Abase + (uint32_t)(kG * PW + g) * 8u);
            const int ob = lds_s32(Bbase + (uint32_t)(kG * PW + ibb[q]) * 8u);
            const int ol = lds_s32(Bbase + (uint32_t)(kG * PW + ibl[q]) * 8u + 4u);
            const int db = min(max(oa.x + ob - EP, -2047), 2047), dl = min(max(oa.y + ol - EP, -2047), 2047);
            dsb[q] = g <= Lb ? db * (1 << 20) : INT_MIN;
            dsl[q] = g < Lb ? dl * (1 << 20) : INT_MIN;
        }
        // Two frames per loop trip (compact code: the CTA's roles share the instruction cache): occupancies of the
        // label states to their rank slots, inclusive prefix sums over the rank order, per symbol the difference of
        // two prefix sums (its run is contiguous in rank order; summation order fixed, no atomics), gradient rows.
#pragma unroll 1
        for (int j2 = 0; j2 < ns; j2 += 2) {
            float nxa[2], nxb[2];
#pragma unroll
            for (int f = 0; f < 2; ++f) {
                const int j = j2 + 2 + f;
                const float* row = xbase + (long long)(t0 + j) * p.st_t;
                nxa[f] = (j < ns && has0) ? __ldg(row + v0) : 0.0f;
                nxb[f] = (j < ns && has1) ? __ldg(row + v1) : 0.0f;
            }
            int2 ha[2][P]; int hbb[2][P], hbl[2][P];
#pragma unroll
            for (int f = 0; f < 2; ++f) {
                const int j = min(j2 + f, kG - 1);
                const uint32_t Arow = Abase + (uint32_t)(j * PW) * 8u, Brow = Bbase + (uint32_t)(j * PW) * 8u;
#pragma unroll
                for (int q = 0; q < P; ++q) {
                    ha[f][q] = lds_v2(Arow + (uint32_t)(q * 32 + lane) * 8u);
                    hbb[f][q] = lds_s32(Brow + (uint32_t)ibb[q] * 8u);
                    hbl[f][q] = lds_s32(Brow + (uint32_t)ibl[q] * 8u + 4u);
                }
            }
            float zb[2];
#pragma unroll
            for (int f = 0; f < 2; ++f) {
                zb[f] = 0.0f;
#pragma unroll
                for (int q = 0; q < P; ++q) {
                    const int2 a_ = ha[f][q];
                    // alpha's high word with the block's exponent shift applied: an exact zero stays zero, anything that
                    // leaves the normal range is flushed to zero (hw_normal_or_zero)
                    int tb = a_.x != 0 ? (int)((unsigned)a_.x + (unsigned)dsb[q]) : 0, tl = a_.y != 0 ? (int)((unsigned)a_.y + (unsigned)dsl[q]) : 0;
                    tb = hw_normal_or_zero(tb); tl = hw_normal_or_zero(tl);
                    zb[f] += (float)(__hiloint2double(tb, 0) * __hiloint2double(tb ? hbb[f][q] : 0, 0));
                    const float gl = (float)(__hiloint2double(tl, 0) * __hiloint2double(tl ? hbl[f][q] : 0, 0));
                    sts_f32(rowbuf + (uint32_t)(f * PW + rk[q]) * 4u, gl);
                }
            }
            __syncwarp();
            // inclusive prefix sums over the rank order: P consecutive slots per lane, then a warp scan of the lane totals
            float sc[2][P];
#pragma unroll
            for (int f = 0; f < 2; ++f) {
#pragma unroll
                for (int q = 0; q < P; ++q) sc[f][q] = lds_f32(rowbuf + (uint32_t)(f * PW + lane * P + q) * 4u);
#pragma unroll
                for (int q = 1; q < P; ++q) sc[f][q] += sc[f][q - 1];
            }
            {
                float t0_ = sc[0][P - 1], t1_ = sc[1][P - 1];
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const float y0 = __shfl_up_sync(FULL, t0_, o), y1 = __shfl_up_sync(FULL, t1_, o);
                    if (lane >= o) { t0_ += y0; t1_ += y1; }
                }
                float e0 = __shfl_up_sync(FULL, t0_, 1), e1 = __shfl_up_sync(FULL, t1_, 1);      // exclusive lane offsets
                if (lane == 0) { e0 = 0.0f; e1 = 0.0f; }
#pragma unroll
                for (int q = 0; q < P; ++q) {
                    sts_f32(sumbuf + (uint32_t)(lane * P + q) * 4u, sc[0][q] + e0);
                    sts_f32(sumbuf + (uint32_t)(PW + lane * P + q) * 4u, sc[1][q] + e1);
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                zb[0] += __shfl_xor_sync(FULL, zb[0], o);
                zb[1] += __shfl_xor_sync(FULL, zb[1], o);
            }
            __syncwarp();
#pragma unroll
            for (int f = 0; f < 2; ++f) {
                const int j = j2 + f;
                if (j < ns) {
                    const uint32_t sb_ = sumbuf + (uint32_t)(f * PW) * 4u;
                    float occ0 = 0.0f, occ1 = 0.0f;
                    if (run0.y > run0.x) occ0 = lds_f32(sb_ + (uint32_t)(run0.y - 1) * 4u) - (run0.x > 0 ? lds_f32(sb_ + (uint32_t)(run0.x - 1) * 4u) : 0.0f);
                    if (run1.y > run1.x) occ1 = lds_f32(sb_ + (uint32_t)(run1.y - 1) * 4u) - (run1.x > 0 ? lds_f32(sb_ + (uint32_t)(run1.x - 1) * 4u) : 0.0f);
                    const float2 fr_ = frr[(blk % kMeetFR) * kG + j];
                    float* grow = grad_b + (long long)(t0 + j) * p.gst_t;
                    if (has0) {
                        const float occ = occ0 + (v0 == c.blank ? zb[f] : 0.0f);
                        const float y = fast_ex2(fmaf(xa[f] - fr_.x, kLog2e, -fr_.y));
                        grow[v0] = head * (y - occ * rP);
                    }
                    if (has1) {
                        const float occ = occ1 + (v1 == c.blank ? zb[f] : 0.0f);
                        const float y = fast_ex2(fmaf(xb[f] - fr_.x, kLog2e, -fr_.y));
                        grow[v1] = head * (y - occ * rP);
                    }
                }
            }
            __syncwarp();
#pragma unroll
            for (int f = 0; f < 2; ++f) { xa[f] = nxa[f]; xb[f] = nxb[f]; }
        }
        MEET_TP(n, 3);
        if (lane == 0) {
            mbar_arrive(c.emptyH(SIDE, h));
            if (n + 2 < NQ) fetch(n + 2);
        }
        __syncwarp();
        MEET_TP(n, 4);
    }
}

template <int P>
__global__ void __launch_bounds__(256, 2) k_meet(MeetArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int PW = 32 * P;
    const Problem& p = a.p;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    __shared__ int s_L, s_rep, s_flags;
    MeetCtx c;
    c.m = meet_smem_layout(P, p.V, (p.Lmax + 3) & ~3);
    c.smem = smem_raw; c.base = smem_u32(smem_raw);
    c.bars = reinterpret_cast<uint64_t*>(smem_raw + c.m.bars);
    c.b = b; c.V = p.V; c.blank = p.blank; c.trace = a.trace;
    if (tid == 0) {
        s_L = p.Lmax; s_rep = 0; s_flags = 0;
        for (int d = 0; d < 2; ++d) {
            for (int s = 0; s < kMeetES; ++s) { mbar_init(c.fullE(d, s), 1); mbar_init(c.emptyE(d, s), 1); }
            for (int s = 0; s < 2; ++s) { mbar_init(c.fullH(d, s), 1); mbar_init(c.emptyH(d, s), 1); mbar_init(c.fullO(d, s), 1); }
            mbar_init(c.HD(d), 2);
        }
        mbar_init(c.J(), 1); mbar_init(c.J2(), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (tid < 2) reinterpret_cast<double*>(smem_raw + c.m.lzp)[tid] = 0.0;
    __syncthreads();
    // ---- operator parameter layer (rows a3/a5), as k_walk's fused prologue ----
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
        for (int j = tid; j < p.Lmax; j += 256)
            if (load_as_int(p.labels, p.label_dtype, b * p.lst_b + j * p.lst_l) == p.label_pad) atomicMin(&s_L, j);
        __syncthreads();
        L = s_L;
    }
    int* slab = reinterpret_cast<int*>(smem_raw + c.m.lab);
    {
        int bad = 0;
        for (int j = tid; j < L; j += 256) {
            long long v = load_as_int(p.labels, p.label_dtype, b * p.lst_b + j * p.lst_l);
            if (v < 0 || v >= p.V || v == p.blank) bad = 1;
            slab[j] = (int)(v < 0 ? 0 : (v >= p.V ? p.V - 1 : v));
        }
        if (bad) atomicOr(&s_flags, UTT_BAD_LABEL);
    }
    __syncthreads();
    {
        int rep = 0;
        for (int j = tid + 1; j < L; j += 256) rep += slab[j] == slab[j - 1];
        if (rep) atomicAdd(&s_rep, rep);
    }
    if (warp == 7) {
        // ranks in the order (label value, position) and the run of every value: two counting passes (V <= 64)
        int* rank = reinterpret_cast<int*>(smem_raw + c.m.rank);
        int2* runv = reinterpret_cast<int2*>(smem_raw + c.m.runv);
        int c0 = 0, c1 = 0;
        for (int j = 0; j < L; ++j) { const int v = slab[j]; c0 += v == lane; c1 += v == lane + 32; }
        int i0 = c0, i1 = c1;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y0 = __shfl_up_sync(0xffffffffu, i0, o), y1 = __shfl_up_sync(0xffffffffu, i1, o);
            if (lane >= o) { i0 += y0; i1 += y1; }
        }
        const int tot0 = __shfl_sync(0xffffffffu, i0, 31);
        int r0 = i0 - c0, r1 = tot0 + i1 - c1;
        runv[lane] = make_int2(r0, r0 + c0);
        runv[lane + 32] = make_int2(r1, r1 + c1);
        for (int j = 0; j < L; ++j) {
            const int v = slab[j];
            if (v == lane) rank[j] = r0++;
            else if (v == lane + 32) rank[j] = r1++;
        }
    }
    __syncthreads();
    int flags = s_flags | lenflags;
    if (Tb <= 0 || L + s_rep > Tb) flags |= UTT_INFEASIBLE;
    if (tid == 0 && p.status && flags) atomicOr(p.status + b, flags);
    if (flags & UTT_INFEASIBLE) {
        // defined behaviour (SURVEY 7.3-6): loss 0, gradient 0
        if (tid == 0) p.loss[b] = 0.0f;
        float* grad_b = p.grad + b * p.gst_b;
        for (int t = warp; t < p.T; t += 8) {
            float* grow = grad_b + (long long)t * p.gst_t;
            for (int v = lane; v < p.V; v += 32) grow[v] = 0.0f;
        }
        return;
    }
    c.Tb = Tb; c.Lb = L;
    c.NQ = (Tb + kG - 1) / kG;
    c.rlast = Tb - (c.NQ - 1) * kG;
    c.NA = (c.NQ + 1) / 2;
    int2* hist_b = a.hist + (size_t)b * a.NB * kHR * PW;
    switch (warp) {
        case 0: case 1: meet_walker<P>(c, p, warp); break;     // one copy of the code for both directions
        case 6: case 7: meet_producer(c, p, warp - 6); break;
        default: meet_helper<P>(c, p, hist_b, warp & 1, (warp - 2) >> 1); break;   // 2, 4: alpha side; 3, 5: beta side
    }
}

}  // namespace ctcb
