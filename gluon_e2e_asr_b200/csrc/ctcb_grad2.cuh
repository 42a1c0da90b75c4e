// ctcb_grad2.cuh -- k_grad2<VEC,CH>: the gradient kernel of the small-vocabulary (fused, V <= 64) path, rows
// a7/a8 of SURVEY.md section 8a (beta + per-label accumulation + gradient + head-gradient scaling of
// `mx.nd.contrib.ctc_loss`, /root/reference/scripts/swbd/loss.py:134-139).  Same launch shape, dispatch order
// and progress protocol as k_grad (one frame block per CTA, blocks of an utterance from the middle outwards,
// concurrent with the walkers), but a third of its instructions per frame (ncu at cfg5: k_grad executes ~690
// warp instructions per frame, half of them integer decode of the stored high words):
//
//   * P(l|x) = sum_s alpha_t(s) beta'_t(s) holds for EVERY frame, so the utterance's middle frame block -- the
//     first one both walkers reach, and the first CTA of the utterance to be dispatched -- forms it once from
//     its first frame (exact integer exponents, fp64 sum) and publishes {exponent, 1/mantissa}; every block
//     then normalises by that one number.  A state's occupancy is: integer add of the block's exponent shift
//     (offset_alpha + offset_beta - exponent of P) on alpha's stored high word, one DMUL with beta's, one
//     conversion -- no mantissa/exponent decode, no per-frame maximum, no per-frame sum of the label states;
//   * the label occupancies, written at their rank in the order (symbol, position), are summed per symbol as
//     the difference of two inclusive prefix sums over the rank order (one warp scan per frame; fixed
//     summation order, no atomics), and the symbol's column of the dense row takes its occupancy in the same
//     pass that writes the row: no second visit of the label columns, no second softmax evaluation.
#pragma once
#include "ctcb_kernels.cuh"

namespace ctcb {

__host__ __device__ inline size_t grad2_smem_bytes(int CH) { return (size_t)4 * 2 * 2 * 32 * CH * 4 + 64 * 8; }

// OCC = 1: 6 CTAs per SM (80 registers); OCC = 0: 7 CTAs per SM (72 registers, a few spilled words)
template <int VEC, int CH, int OCC, typename LT = float>
__global__ void __launch_bounds__(128, CH <= 4 ? (OCC ? 6 : 7) : (CH == 8 ? 4 : 2)) k_grad2(GradArgs a) {
    using V_t = typename LV<LT, VEC>::type;
    constexpr int FPW = kGradFramesPerWarp;               // 2 frames per warp, 4 warps: one frame block per trip
    constexpr int F = CH <= 4 ? FPW : 1;                  // frames in flight per warp
    constexpr int GW = 32 * CH;                           // rank slots per frame
    constexpr int NXQ = 64 / (32 * VEC) > 0 ? 64 / (32 * VEC) : 1;   // vector loads per lane that cover a row of V <= 64
    constexpr unsigned FULL = 0xffffffffu;
    const Problem& p = a.p; const Workspace& w = a.w;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    __shared__ int s_ok, s_EP; __shared__ float s_rP;
    extern __shared__ __align__(128) unsigned char g2sm[];
    float* gbuf0 = reinterpret_cast<float*>(g2sm) + (size_t)warp * (2 * FPW * GW);    // per warp: [FPW][GW] gamma, [FPW][GW] prefix sums
    int2* s_run = reinterpret_cast<int2*>(g2sm + (size_t)4 * 2 * FPW * GW * 4);       // [64] runs of the symbols
    // A CTA takes G consecutive frame blocks of its utterance in the middle-outwards order (the order the walkers
    // complete them): metadata, the symbols' runs and P(l|x) are fetched once per CTA, not once per frame block
    const int G = (w.NB + (int)gridDim.y - 1) / (int)gridDim.y;
    if (tid == 0) {
        const long long t0 = clock64();
        int v;
        while ((v = ld_acquire_gpu(w.gprog + 4 * b + 2)) == 0 && clock64() - t0 < kSpinLimit) __nanosleep(256);
        s_ok = v == w.stamp;
    }
    __syncthreads();
    auto nan_rows = [&](int t_first, int t_end) {            // a workspace no matching forward call filled: NaN, not a hang
        for (int t = t_first + warp; t < t_end && t < p.T; t += 4) {
            LT* grow = grad_row<LT>(p, b, t);
            for (int v = lane; v < p.V; v += 32) stx(grow + v, __int_as_float(0x7fc00000));
        }
    };
    if (!s_ok) { for (int i = 0; i < G; ++i) { const int vi = blockIdx.y * G + i; if (vi < w.NB) nan_rows(vi * kG, vi * kG + kG); } return; }
    const int Tb = __ldcg(w.Tb + b), Lb = __ldcg(w.Lb + b);
    const bool infeasible = (__ldcg(w.flags + b) & UTT_INFEASIBLE) != 0;
    const int NQ = infeasible ? 0 : (Tb + kG - 1) / kG;
    auto block_of = [&](int vi) { return vi < NQ ? ((vi & 1) ? NQ / 2 - (vi + 1) / 2 : NQ / 2 + vi / 2) : vi; };
    const float head = p.head ? p.head[b] : 1.0f;
    const int pairs = 32 * w.P * w.NW;
    const int* gp = w.gprog + 4 * b;
    // both walkers are past frame block blk (bounded wait; lane 0 polls for its warp)
    auto wait_block = [&](int blk) -> bool {
        int ok = 1;
        if (lane == 0) {
            const long long t0 = clock64();
            const unsigned pns = w.poll_ns > 0 ? (unsigned)w.poll_ns : 128u;
            while (ld_acquire_gpu(gp) < blk + 1 && clock64() - t0 < kSpinLimit) __nanosleep(pns);
            while (ld_acquire_gpu(gp + 1) < NQ - blk && clock64() - t0 < kSpinLimit) __nanosleep(pns);
            ok = clock64() - t0 < kSpinLimit;
        }
        return __shfl_sync(FULL, ok, 0) != 0;
    };
    const bool cta_live = blockIdx.y * G < NQ;             // at least one of this CTA's blocks holds frames of the utterance
    if (cta_live && tid < 64) s_run[tid] = tid < p.V ? __ldcg(w.runv + (size_t)b * 64 + tid) : make_int2(0, 0);
    if (cta_live && blockIdx.y == 0 && warp == 0) {
        // ---- the utterance's middle block: P(l|x) from its first frame, once for all blocks ----
        const int blk = block_of(0);
        const size_t blkoff = (size_t)b * w.NB + blk;
        const int2* hA0 = w.hA + blkoff * kG * pairs;
        const int2* hB0 = w.hB + blkoff * kG * pairs;
        const int2* oA = w.oA + blkoff * pairs;
        const int2* oB = w.oB + blkoff * pairs;
        if (wait_block(blk)) {
            int ex[2 * CH]; float mm[2 * CH];
            int emax = INT_MIN / 2;
#pragma unroll
            for (int c = 0; c < CH; ++c) {
                const int g = c * 32 + lane;
                const int ib = max(Lb - g, 0), il = max(Lb - 1 - g, 0);
                const int2 av = __ldcg(hA0 + g), oa = __ldcg(oA + g);
                const int hb = __ldcg(&hB0[ib].x), hl = __ldcg(&hB0[il].y);
                const int ob = __ldcg(&oB[ib].x), ol = __ldcg(&oB[il].y);
                const bool vb = g <= Lb && av.x != 0 && hb != 0, vl = g < Lb && av.y != 0 && hl != 0;
                ex[2 * c] = vb ? (av.x >> 20) + (hb >> 20) - 2046 + oa.x + ob : INT_MIN / 2;
                ex[2 * c + 1] = vl ? (av.y >> 20) + (hl >> 20) - 2046 + oa.y + ol : INT_MIN / 2;
                mm[2 * c] = vb ? hw_mant(av.x) * hw_mant(hb) : 0.0f;
                mm[2 * c + 1] = vl ? hw_mant(av.y) * hw_mant(hl) : 0.0f;
                emax = max(emax, max(ex[2 * c], ex[2 * c + 1]));
            }
            emax = __reduce_max_sync(FULL, emax);
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < 2 * CH; ++k) s += (double)mm[k] * pow2c(max(ex[k] - emax, -2000));
#pragma unroll
            for (int o = 16; o > 0; o >>= 1)
                s += __hiloint2double(__shfl_xor_sync(FULL, __double2hiint(s), o), __shfl_xor_sync(FULL, __double2loint(s), o));
            if (lane == 0) {
                const int EP = emax + dexp(s);
                const float rP = (float)(1.0 / dmant(s));
                w.pinfo[b] = make_int2(EP, __float_as_int(rP));
                __threadfence();
                st_release_gpu(w.gprog + 4 * b + 3, w.stamp);
            }
        }
    }
    if (cta_live && tid == 0) {
        const long long t0 = clock64();
        int v;
        while ((v = ld_acquire_gpu(w.gprog + 4 * b + 3)) != w.stamp && clock64() - t0 < kSpinLimit) __nanosleep(128);
        if (v != w.stamp) s_ok = 0;
        const int2 pi = __ldcg(w.pinfo + b);
        s_EP = pi.x; s_rP = __int_as_float(pi.y);
    }
    __syncthreads();
    if (!s_ok) { for (int i = 0; i < G; ++i) { const int vi = blockIdx.y * G + i; if (vi < w.NB) nan_rows(block_of(vi) * kG, block_of(vi) * kG + kG); } return; }
    const int EP = s_EP; const float rP = s_rP;

    // per lane and chunk, once per CTA: history indices of the reversed walker, rank slots
    const int* rank = w.rank + (size_t)b * w.Lp;
    int ibb[CH], ibl[CH], rk[CH];
#pragma unroll
    for (int c = 0; c < CH; ++c) {
        const int g = c * 32 + lane;
        ibb[c] = max(Lb - g, 0); ibl[c] = max(Lb - 1 - g, 0);
        rk[c] = (cta_live && g < Lb) ? __ldcg(rank + g) : g;
    }
    // the runs of this lane's symbols (column k*VEC + j of vector k = q*32 + lane)
    const int nvec = p.V / VEC;
    int2 run[NXQ][VEC];
#pragma unroll
    for (int q = 0; q < NXQ; ++q)
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            const int v = (q * 32 + lane) * VEC + j;
            run[q][j] = (cta_live && v < p.V) ? s_run[v] : make_int2(0, 0);
        }

    // ---- the CTA's frame blocks; no CTA barrier from here on: every warp waits for its blocks itself ----
    // A warp takes WHOLE frame blocks (all kG frames, F at a time): the block's exponent shifts are formed once per
    // kG frames, not once per two (ncu at cfg5: the per-block part was 130 of 490 instructions per frame)
#pragma unroll 1
    for (int i = warp; i < G; i += 4) {
        const int vi = blockIdx.y * G + i;
        if (vi >= w.NB) break;
        const int blk = block_of(vi);
        const int t_first = blk * kG;
        const bool blk_live = blk < NQ;
        const size_t blkoff = (size_t)b * w.NB + blk;
        const int2* hA0 = w.hA + blkoff * kG * pairs;
        const int2* hB0 = w.hB + blkoff * kG * pairs;
        const int2* oA = w.oA + blkoff * pairs;
        const int2* oB = w.oB + blkoff * pairs;
        int dsb[CH], dsl[CH];
        if (blk_live) {
            if (!wait_block(blk)) {
                for (int t = t_first; t < t_first + kG && t < p.T; ++t) {
                    LT* grow = grad_row<LT>(p, b, t);
                    for (int v = lane; v < p.V; v += 32) stx(grow + v, __int_as_float(0x7fc00000));
                }
                continue;
            }
            // exponent shifts of the block's states: offsets of both directions minus the exponent of P(l|x)
#pragma unroll
            for (int c = 0; c < CH; ++c) {
                const int g = c * 32 + lane;
                const int2 oa = __ldcg(oA + g);
                const int ob = __ldcg(&oB[ibb[c]].x), ol = __ldcg(&oB[ibl[c]].y);
                const int db = min(max(oa.x + ob - EP, -2047), 2047), dl = min(max(oa.y + ol - EP, -2047), 2047);
                dsb[c] = g <= Lb ? db * (1 << 20) : INT_MIN;
                dsl[c] = g < Lb ? dl * (1 << 20) : INT_MIN;
            }
        }
#pragma unroll 1
        for (int r = 0; r < kG / F; ++r) {
            int tt[F]; bool live[F];
            int2 ha[F][CH <= 4 ? CH : 1], hb2[F][CH <= 4 ? CH : 1];
            V_t xr[F][NXQ]; float2 fr[F];
            // ---- every global load of the F frames ----
#pragma unroll
            for (int f = 0; f < F; ++f) {
                tt[f] = t_first + r * F + f;
                live[f] = blk_live && tt[f] < Tb;
                fr[f] = make_float2(0.0f, 0.0f);
                if (live[f]) {
                    fr[f] = __ldcg(w.fr + (size_t)b * p.T + tt[f]);
                    const V_t* xv = reinterpret_cast<const V_t*>(utt_logits<LT>(p, b) + (long long)tt[f] * p.st_t);
#pragma unroll
                    for (int q = 0; q < NXQ; ++q) { const int k = q * 32 + lane; xr[f][q] = k < nvec ? __ldg(xv + k) : LV<LT, VEC>::fill(0.0f); }
                    if (CH <= 4) {
                        const int2* A = hA0 + (size_t)(tt[f] - t_first) * pairs + lane;
                        const int2* Bh = hB0 + (size_t)(tt[f] - t_first) * pairs;
#pragma unroll
                        for (int c = 0; c < (CH <= 4 ? CH : 1); ++c) {
                            ha[f][c] = __ldcg(A + c * 32);
                            hb2[f][c] = __ldcg(Bh + ibb[c]);       // {blank of slot L-g, label of slot L-g}: ONE 8-byte load
                        }
                    }
                }
            }
#pragma unroll
            for (int f = 0; f < F; ++f) {
                const int t = tt[f];
                if (t >= p.T) continue;
                LT* grow = grad_row<LT>(p, b, t);
                if (!live[f]) { zero_row<VEC>(grow, p.V, lane); continue; }
                float* gbuf = gbuf0 + (size_t)f * GW;                       // gamma of the label states, rank order
                float* sbuf = gbuf0 + (size_t)(FPW + f) * GW;               // inclusive prefix sums
                float zb = 0.0f;
                auto occupancy = [&](int2 av, int hb, int hl, int c) {
                    // alpha's high word with the block's exponent shift applied: an exact zero stays zero, anything that leaves
                    // the normal range (an occupancy below 2^-1022 times the largest beta') is flushed to zero
                    int tb = av.x != 0 ? (int)((unsigned)av.x + (unsigned)dsb[c]) : 0, tl = av.y != 0 ? (int)((unsigned)av.y + (unsigned)dsl[c]) : 0;
                    tb = tb < (1 << 20) ? 0 : tb; tl = tl < (1 << 20) ? 0 : tl;
                    zb += (float)(__hiloint2double(tb, 0) * __hiloint2double(tb ? hb : 0, 0));
                    gbuf[rk[c]] = (float)(__hiloint2double(tl, 0) * __hiloint2double(tl ? hl : 0, 0));
                };
                if (CH <= 4) {
                    // the label state of slot L-1-g is the label word the lane ABOVE loaded (its g is one higher; the
                    // clamped indices agree: max(L-(g+1), 0) = max(L-1-g, 0)); lane 31 takes it from the next chunk's lane 0
#pragma unroll
                    for (int c = 0; c < (CH <= 4 ? CH : 1); ++c) {
                        int hl = __shfl_down_sync(FULL, hb2[f][c].y, 1);
                        if (c + 1 < (CH <= 4 ? CH : 1)) { const int nx = __shfl_sync(FULL, hb2[f][c + 1 < (CH <= 4 ? CH : 1) ? c + 1 : c].y, 0); if (lane == 31) hl = nx; }
                        occupancy(ha[f][c], hb2[f][c].x, hl, c);
                    }
                } else {
                    const int2* A = hA0 + (size_t)(t - t_first) * pairs + lane;
                    const int2* Bh = hB0 + (size_t)(t - t_first) * pairs;
#pragma unroll
                    for (int c0 = 0; c0 < CH; c0 += 4) {
                        int2 av[4]; int hb[4], hl[4];
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            // lanes past the walkers' 32 * P * NW pairs (8 or 16 chunks cover more) hold no state: a load
                            // there would read the next frame's row, never written past T_b, and a word with its sign bit
                            // set wraps to a positive value under the INT_MIN shift of a state beyond the lattice
                            av[k] = (c0 + k) * 32 + lane < pairs ? __ldcg(A + (c0 + k) * 32) : make_int2(0, 0);
                            hb[k] = __ldcg(&Bh[ibb[c0 + k]].x); hl[k] = __ldcg(&Bh[ibl[c0 + k]].y);
                        }
#pragma unroll
                        for (int k = 0; k < 4; ++k) occupancy(av[k], hb[k], hl[k], c0 + k);
                    }
                }
                zb = warp_sum(zb);
                __syncwarp();
                // inclusive prefix sums over the rank order: CH consecutive slots per lane, then a warp scan of the lane totals
                {
                    float sc[CH];
#pragma unroll
                    for (int c = 0; c < CH; ++c) sc[c] = gbuf[lane * CH + c];
#pragma unroll
                    for (int c = 1; c < CH; ++c) sc[c] += sc[c - 1];
                    float tot = sc[CH - 1];
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) { const float y = __shfl_up_sync(FULL, tot, o); if (lane >= o) tot += y; }
                    float ex_ = __shfl_up_sync(FULL, tot, 1);            // exclusive: the lanes below (slots past the labels may hold anything)
                    if (lane == 0) ex_ = 0.0f;
#pragma unroll
                    for (int c = 0; c < CH; ++c) sbuf[lane * CH + c] = sc[c] + ex_;
                }
                __syncwarp();
                const float fmx = fr[f].x, flz = fr[f].y;
                V_t* gv = reinterpret_cast<V_t*>(grow);
#pragma unroll
                for (int q = 0; q < NXQ; ++q) {
                    const int k = q * 32 + lane;
                    if (k < nvec) {
                        float x[VEC]; LV<LT, VEC>::get(xr[f][q], x);
                        float y[VEC];
#pragma unroll
                        for (int j = 0; j < VEC; ++j) {
                            const int2 rn = run[q][j];
                            float occ = 0.0f;
                            if (rn.y > rn.x) occ = sbuf[rn.y - 1] - (rn.x > 0 ? sbuf[rn.x - 1] : 0.0f);
                            if (k * VEC + j == p.blank) occ += zb;
                            y[j] = head * (fast_ex2(fmaf(x[j] - fmx, kLog2e, -flz)) - occ * rP);
                        }
                        gv[k] = LV<LT, VEC>::pack(y);
                    }
                }
                __syncwarp();
            }
        }
    }
    // the stream's next kernel must also see what the walkers write last (loss, loss_sum)
    if (blockIdx.x == 0 && blockIdx.y == 0 && tid == 0) asm volatile("griddepcontrol.wait;" ::: "memory");
}

}  // namespace ctcb
