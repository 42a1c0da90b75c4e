/* TEST INFRASTRUCTURE ONLY -- body of oracle/ctc_ref.c, included once per REAL type.
 * See that file's header for scope, provenance and the parity statement. */

#define NEGINF ((REAL)(-INFINITY))

static inline REAL CAT(log_add_, SUFFIX)(REAL a, REAL b) {
    if (a == NEGINF) return b;
    if (b == NEGINF) return a;
    return a > b ? a + (REAL)log1p(EXP(b - a)) : b + (REAL)log1p(EXP(a - b));
}

/* One utterance.  x/g address frame t at x + t*st_t (V contiguous).  Returns 0 when the
 * alignment is infeasible (cost 0, gradient 0 -- SURVEY.md 7.3-6), 1 otherwise. */
static int CAT(one_utt_, SUFFIX)(const REAL* x, long st_t, REAL* g, long gst_t,
                                 const int* lab, int L, int Tb, int V, int blank,
                                 REAL head, REAL* cost) {
    const int S = 2 * L + 1;
    int repeats = 0;
    for (int i = 1; i < L; ++i) repeats += (clamp_label(lab[i], V) == clamp_label(lab[i - 1], V));
    *cost = 0;
    if (Tb <= 0 || L + repeats > Tb) return 0;

    REAL* probs = (REAL*)malloc(sizeof(REAL) * ((size_t)Tb * V + (size_t)Tb * S + 2 * (size_t)S + V));
    REAL* alphas = probs + (size_t)Tb * V;
    REAL* beta_cur = alphas + (size_t)Tb * S;
    REAL* beta_nxt = beta_cur + S;
    REAL* acc = beta_nxt + S;
    int* ext = (int*)malloc(sizeof(int) * 2 * (size_t)S);
    int* skip = ext + S;   /* skip[s] = 1 when the s-2 -> s transition is allowed */

    /* labels clamped to [0, V-1]; a skip into a state is allowed exactly when its symbol differs from the one two
     * states back (a label equal to the blank is a state of its own, as in torch's ctc_loss) */
    for (int s = 0; s < S; ++s) ext[s] = (s & 1) ? clamp_label(lab[s / 2], V) : blank;
    for (int s = 0; s < S; ++s) skip[s] = (s >= 2 && ext[s] != ext[s - 2]);

    /* a4: softmax in probability space */
    for (int t = 0; t < Tb; ++t) {
        const REAL* row = x + t * st_t;
        REAL* p = probs + (size_t)t * V;
        REAL mx = row[0];
        for (int v = 1; v < V; ++v) mx = row[v] > mx ? row[v] : mx;
        REAL den = 0;
        for (int v = 0; v < V; ++v) { p[v] = EXP(row[v] - mx); den += p[v]; }
        for (int v = 0; v < V; ++v) p[v] /= den;
    }

    /* a6: alpha, log space, only the band of states that can still reach the end */
    for (size_t i = 0; i < (size_t)Tb * S; ++i) alphas[i] = NEGINF;
    alphas[0] = LOG(probs[blank]);
    if (S > 1) alphas[1] = LOG(probs[ext[1]]);
    for (int t = 1; t < Tb; ++t) {
        int lo = S - 2 * (Tb - t); if (lo < 0) lo = 0;
        int hi = 2 * (t + 1);      if (hi > S) hi = S;
        const REAL* prev = alphas + (size_t)(t - 1) * S;
        REAL* cur = alphas + (size_t)t * S;
        const REAL* p = probs + (size_t)t * V;
        for (int s = lo; s < hi; ++s) {
            REAL a = prev[s];
            if (s >= 1) a = CAT(log_add_, SUFFIX)(a, prev[s - 1]);
            if (skip[s]) a = CAT(log_add_, SUFFIX)(a, prev[s - 2]);
            cur[s] = a + LOG(p[ext[s]]);
        }
    }
    REAL loglik = alphas[(size_t)(Tb - 1) * S + S - 1];
    if (S > 1) loglik = CAT(log_add_, SUFFIX)(loglik, alphas[(size_t)(Tb - 1) * S + S - 2]);
    *cost = -loglik;
    if (!g) { free(probs); free(ext); return 1; }

    /* a7: beta fused with the per-label accumulation and the gradient */
    for (int t = Tb - 1; t >= 0; --t) {
        const REAL* p = probs + (size_t)t * V;
        REAL* al = alphas + (size_t)t * S;
        int lo = S - 2 * (Tb - t); if (lo < 0) lo = 0;
        int hi = 2 * (t + 1);      if (hi > S) hi = S;
        for (int s = 0; s < S; ++s) beta_cur[s] = NEGINF;
        if (t == Tb - 1) {
            beta_cur[S - 1] = LOG(p[blank]);
            if (S > 1) beta_cur[S - 2] = LOG(p[ext[S - 2]]);
        } else {
            for (int s = lo; s < hi; ++s) {
                REAL b = beta_nxt[s];
                if (s + 1 < S) b = CAT(log_add_, SUFFIX)(b, beta_nxt[s + 1]);
                if (s + 2 < S && skip[s + 2]) b = CAT(log_add_, SUFFIX)(b, beta_nxt[s + 2]);
                beta_cur[s] = b + LOG(p[ext[s]]);
            }
        }
        for (int v = 0; v < V; ++v) acc[v] = NEGINF;
        for (int s = lo; s < hi; ++s)
            acc[ext[s]] = CAT(log_add_, SUFFIX)(acc[ext[s]], al[s] + beta_cur[s]);
        REAL* grow = g + t * gst_t;
        for (int v = 0; v < V; ++v) {
            REAL gv;
            if (acc[v] == NEGINF || p[v] == 0) gv = p[v];
            else gv = p[v] - EXP(acc[v] - LOG(p[v]) - loglik);
            grow[v] = head * gv;       /* a8 */
        }
        REAL* tmp = beta_cur; beta_cur = beta_nxt; beta_nxt = tmp;
    }
    free(probs); free(ext);
    return 1;
}

/* Batch entry.  acts/grads: element strides (st_t, st_b), V contiguous, so both the
 * operator's TNC layout and the model's NTC layout can be addressed.  labels: (B, Lmax)
 * int32.  grads may be NULL (forward only).  head_grad may be NULL (= 1).  feasible may
 * be NULL.  Padded frames t >= input_lengths[b] get gradient 0. */
int CAT(ctc_ref_loss_grad_, SUFFIX)(const REAL* acts, long st_t, long st_b,
                                    REAL* grads, long gst_t, long gst_b,
                                    const int* labels, int Lmax,
                                    const int* label_lengths, const int* input_lengths,
                                    const REAL* head_grad, int T, int B, int V, int blank,
                                    REAL* costs, int* feasible, int num_threads) {
    if (!acts || !labels || !label_lengths || !input_lengths || !costs) return 1;
    if (blank < 0 || blank >= V) return 1;
#ifdef _OPENMP
    if (num_threads > 0) omp_set_num_threads(num_threads);
#endif
#pragma omp parallel for schedule(dynamic, 1)
    for (int b = 0; b < B; ++b) {
        int Tb = input_lengths[b]; if (Tb > T) Tb = T; if (Tb < 0) Tb = 0;
        int L = label_lengths[b];  if (L > Lmax) L = Lmax; if (L < 0) L = 0;
        REAL head = head_grad ? head_grad[b] : (REAL)1;
        REAL* gb = grads ? grads + b * gst_b : NULL;
        int ok = CAT(one_utt_, SUFFIX)(acts + b * st_b, st_t, gb, gst_t,
                                       labels + (size_t)b * Lmax, L, Tb, V, blank, head, costs + b);
        if (feasible) feasible[b] = ok;
        if (gb) {
            int from = ok ? Tb : 0;
            for (int t = from; t < T; ++t) memset(gb + t * gst_t, 0, sizeof(REAL) * V);
        }
    }
    return 0;
}

#undef NEGINF
