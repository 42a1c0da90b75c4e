/* TEST INFRASTRUCTURE ONLY -- C restatement of the reference's CPU CTC operator.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
 * legs may load the library built from this file (oracle/libctc_ref.so).  Nothing under
 * gluon_e2e_asr_b200/ links, loads or calls it.
 *
 * What it restates.  scripts/swbd/loss.py:134-139 calls MXNet's `contrib.ctc_loss`; on
 * `mx.cpu()` that operator is MXNet 1.x's vendored Baidu warp-ctc CPU path (NOT in
 * /root/reference, not installable here, no version pinned by the reference -- see
 * oracle/ctc_oracle.py's header).  This file restates that path's *structure*, written
 * from the published algorithm (SURVEY.md section 8 rows a4-a8), not from its source:
 *
 *   a4  probability-space softmax per valid frame, max-subtracted;
 *   a5  blank-extended label lattice (labels clamped to [0, V-1]), repeats, feasibility
 *       (L + repeats <= T);
 *   a6  log-space alpha recursion with the reachable-band limits;
 *   a7  log-space beta recursion fused with the per-label log-sum-exp of alpha+beta
 *       and  grad = y - exp(acc - log y - loglik);
 *   a8  head-gradient scaling (the operator's backward);
 *   parallelism: one `omp parallel for` over the minibatch, which is how the CPU
 *   operator is parallelised (SURVEY.md section 2.2).
 *
 * It is compiled twice, with REAL = float (the reference-class arithmetic, used as the
 * timed CPU baseline, `kind: "port"`) and REAL = double (a second fp64 opinion for
 * tests/test_oracle.py).  PARITY STATUS: unpinned by the reference itself; pinned by
 * upstream KATs K1-K5 and by agreement with oracle/ctc_oracle.py (tests/test_oracle.py).
 *
 * Build:  make -C oracle        (gcc -O3 -march=x86-64-v3 -fopenmp -shared -fPIC)
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* the operator's label clamp: out-of-range labels become the nearest valid symbol */
static inline int clamp_label(int v, int V) { return v < 0 ? 0 : (v >= V ? V - 1 : v); }

#define CAT_(a, b) a##b
#define CAT(a, b) CAT_(a, b)

#define REAL float
#define SUFFIX f32
#define EXP expf
#define LOG logf
#include "ctc_ref_impl.h"
#undef REAL
#undef SUFFIX
#undef EXP
#undef LOG

#define REAL double
#define SUFFIX f64
#define EXP exp
#define LOG log
#include "ctc_ref_impl.h"
#undef REAL
#undef SUFFIX
#undef EXP
#undef LOG

int ctc_ref_max_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}
