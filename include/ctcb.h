/* ctcb.h -- C ABI of libctcb.so, the B200 (sm_100a) CTC training-loss path.
 *
 * This is the drop-in boundary for ONE path of Hex-Lee/gluon-e2e-asr: the CTC loss
 * forward+backward that scripts/swbd/train_ctc_ce.py:143 and :363 reach through
 * scripts/swbd/loss.py:121-139 (`CtcLoss.hybrid_forward`) ->
 * `mx.nd.contrib.ctc_loss(data, label, data_lengths, label_lengths, use_data_lengths,
 * use_label_lengths, blank_label)`  (loss.py:134-139).  Every entry point below names the
 * reference interface it replaces.  The library has no Python, torch or MXNet types in
 * its signatures: plain pointers, sizes, strides and (optionally) DLPack structs.
 *
 * Conventions
 *   - return 0 (CTCB_OK) on success, a ctcb_status_t otherwise; the message is in
 *     ctcb_last_error() (thread-local).  No exception, abort or host sync crosses the ABI.
 *   - all device entry points are ASYNCHRONOUS: they enqueue on `stream` (a cudaStream_t
 *     passed as void*; NULL = the legacy default stream) and return.  Labels and lengths
 *     are read on the device -- unlike the reference operator there is no D2H copy of
 *     labels/lengths and no `.asscalar()` (train_ctc_ce.py:367-368).
 *   - the caller owns every buffer including the workspace; the library borrows them for
 *     the duration of the enqueued work.
 *   - there is no CPU fallback: a missing CUDA device or non-device pointer is an error.
 */
#ifndef CTCB_H_
#define CTCB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CTCB_VERSION 103 /* 0.1.3: ctcb_proj_forward, ctcb_proj_loss_grad (fp32 / bf16 operands) */

typedef enum {
    CTCB_OK = 0,
    CTCB_INVALID_VALUE = 1,       /* bad dtype / device / shape / stride / alignment / NULL */
    CTCB_WORKSPACE_TOO_SMALL = 2,
    CTCB_EXECUTION_FAILED = 3,    /* a CUDA launch or runtime error */
    CTCB_MEMOPS_FAILED = 4,       /* allocation or copy failed (host-buffer entry only) */
    CTCB_UNSUPPORTED = 5          /* e.g. no sm_100 device, NCCL not loadable */
} ctcb_status_t;

/* element types accepted for labels and lengths: the reference's data pipeline delivers
 * float32 for all three (reader_kaldi_io.py:33-35, gluonE2EASR/data/batchify.py:78-82);
 * values are truncated toward zero like the operator's own cast.
 * CTCB_BF16 is a LOGITS type only (the *_typed entries below); labels and lengths in bfloat16 are refused (integers
 * above 256 are not exact in bfloat16). */
typedef enum { CTCB_I32 = 0, CTCB_I64 = 1, CTCB_F32 = 2, CTCB_F64 = 3, CTCB_BF16 = 4 } ctcb_dtype_t;

/* per-utterance status bits written to ctcb_problem_t.status (optional) */
/* The parameter layer, identical on every kernel path.  Lengths are truncated toward zero, then clamped to [0, T] and
 * [0, Lmax]; labels are truncated toward zero, then clamped to [0, V-1]; an inferred label length (label_lengths NULL)
 * compares the unclamped truncated label with label_pad.  A label equal to the blank is a lattice state of its own that
 * emits with the blank's probability, and the skip into label j is allowed exactly when label j != label j-1 (torch's
 * rule), so every utterance with L + repeats <= T has a finite loss.  NaN labels or lengths have no defined meaning. */
#define CTCB_UTT_INFEASIBLE   1  /* L + repeats > T (or T == 0), repeats of the clamped labels: loss 0, grad 0 (SURVEY 7.3-6) */
#define CTCB_UTT_BAD_LABEL    2  /* one of the first L truncated labels was < 0, >= V or == blank: clamped / kept as a state */
#define CTCB_UTT_LEN_CLAMPED  4  /* a truncated length was < 0, > T or > Lmax: clamped (a fractional length sets nothing) */
#define CTCB_UTT_WIDE_LOGITS  8  /* CONTRACT DIFFERENCE from mx.nd.contrib.ctc_loss: an emission of a valid frame lay
                                  * more than 100 bits (69.3 nats) below the frame's largest softmax numerator and was
                                  * FLOORED there (small vocabularies: any symbol of the frame; wide ones: a blank or
                                  * label column of this utterance).  Loss and gradient are then those of the floored
                                  * lattice (the reference's fp32 log-space operator has its own, lower floor: log y is
                                  * -inf below e^-103).  Never raised for logit ranges below 69 nats per frame. */

/* One CTC problem = one call of the reference operator (loss.py:134-139).
 * All pointers are DEVICE pointers for ctcb_loss_grad(), HOST pointers for
 * ctcb_loss_grad_host().  Strides are in ELEMENTS; the vocabulary axis of logits/grad has
 * stride 1.  layout 'TNC' (the operator's): stride_t = B*V, stride_b = V;
 * layout 'NTC' (the model's, model.py:421-424): stride_t = V, stride_b = T*V -- the
 * reference's materialising swapaxes (loss.py:123-124) and its backward are not needed. */
typedef struct ctcb_problem {
    int32_t T, B, V, Lmax;          /* Lmax = label row length (may be 0) */
    int32_t blank;                  /* 0 for blank_label='first' (loss.py:139), V-1 for 'last' */
    int32_t label_pad;              /* padding value that ends a label row when label_lengths
                                       is NULL: 0 for 'first', -1 for 'last' (row a3) */
    const float* logits;            /* unnormalised activations, fp32 (bf16 through the *_typed entries) */
    int64_t logits_stride_t, logits_stride_b;
    float* grad;                    /* d(sum_b head[b]*loss[b])/d logits, the logits' type; NULL = forward only */
    int64_t grad_stride_t, grad_stride_b;
    const void* labels;             /* (B, Lmax), label_dtype */
    int32_t label_dtype;            /* ctcb_dtype_t */
    int64_t label_stride_b, label_stride_l; /* 'NT': (Lmax, 1); 'TN' (loss.py:125-126): (1, B) */
    const void* data_lengths;       /* (B,) or NULL (= T; use_data_lengths=False) */
    int32_t data_lengths_dtype;
    const void* label_lengths;      /* (B,) or NULL (= first label_pad; use_label_lengths=False) */
    int32_t label_lengths_dtype;
    const float* head_grad;         /* (B,) upstream gradient of each loss, NULL = 1 */
    float* loss;                    /* (B,) negative log-likelihood per utterance */
    double* loss_sum;               /* optional device scalar: += sum_b loss[b] (feeds the
                                       loss-sum allreduce, replaces train_ctc_ce.py:367-368) */
    int32_t* status;                /* optional (B,) CTCB_UTT_* bits */
    const int64_t* logits_row_offsets; /* optional (B,): PACKED logits -- utterance b's frame 0 is at logits +
                                       logits_row_offsets[b] (elements), its frames logits_stride_t apart, and only its
                                       data_lengths[b] valid frames need to exist: a length-bucketed batch
                                       (data/sampler.py:80-248) crosses PCIe without its padded frames
                                       (batch.py PinnedBatch(packed=True)).  Replaces b * logits_stride_b, which is
                                       then ignored.  Needs data_lengths.  The gradient stays dense (grad strides).
                                       Device pointer for the device entries, host pointer for the host entries. */
} ctcb_problem_t;

/* library identity; replaces nothing (sanity check for the binding) */
int ctcb_version(void);
const char* ctcb_last_error(void);

/* Workspace the caller must provide for a (T,B,V,Lmax) problem.  need_grad=0 sizes the
 * forward-only (evaluation, train_ctc_ce.py:143) path.  Precedent: warp-ctc's
 * get_workspace_size(). */
int ctcb_workspace_bytes(int32_t T, int32_t B, int32_t V, int32_t Lmax, int32_t need_grad,
                         size_t* out_bytes);

/* The operator: loss (and gradient when p->grad != NULL) of one batch, device buffers.
 * Replaces mx.nd.contrib.ctc_loss forward + backward (loss.py:134-139; SURVEY section 8
 * rows a3-a8).  Workspace must be 256-byte aligned device memory. */
int ctcb_loss_grad(const ctcb_problem_t* p, void* workspace, size_t workspace_bytes,
                   void* stream);

/* The same work split the way an autograd engine calls it (MXNet's operator stores its
 * gradient in Forward and scales it in Backward, SURVEY 8a row a8; here Forward keeps the
 * alpha/beta history in the workspace and Backward writes head_grad * G once):
 *   ctcb_forward   loss only (p->grad, p->head_grad ignored).  keep_for_backward != 0 also
 *                  runs the beta walker and keeps the history; the workspace must then be
 *                  sized with need_grad=1 and left untouched until ctcb_backward has run.
 *   ctcb_backward  gradient from a workspace filled by ctcb_forward(keep_for_backward=1) of
 *                  the SAME problem; reads p->head_grad, writes p->grad. */
int ctcb_forward(const ctcb_problem_t* p, int32_t keep_for_backward, void* workspace,
                 size_t workspace_bytes, void* stream);
int ctcb_backward(const ctcb_problem_t* p, void* workspace, size_t workspace_bytes,
                  void* stream);

/* The same three entries with the logits' element type: logits_dtype CTCB_F32 (exactly the entries above, which are these
 * with CTCB_F32) or CTCB_BF16 (a mixed-precision model's logits, read without an upcast pass).  p->logits and p->grad are
 * then read as that type (strides and logits_row_offsets stay in elements); the gradient has the logits' type.
 * The bfloat16 contract:
 *   - a bf16 logit is converted to fp32 exactly when it is loaded; after the load every operation is the fp32 path's, in
 *     the same order, and the kernels selected are those of the fp32 call on the upcast logits (same launches, gradient
 *     kernel and walker configuration).  One exception: the bulk-copy (staged) variants of the wide-vocabulary kernels
 *     need 16-byte aligned rows of a multiple of 16 bytes, so a bf16 call with V % 8 != 0 (or strides not multiples of
 *     8 elements) takes the register variants where the fp32 call with V % 4 == 0 is staged -- same results, other kernels;
 *   - loss (fp32), head_grad (fp32), loss_sum (fp64) and the status word are unchanged: the loss and the status word are
 *     bit-identical to the fp32 call on the upcast logits, CTCB_UTT_WIDE_LOGITS included;
 *   - each gradient element is the fp32 path's value rounded ONCE to bfloat16 (round to nearest even); padded frames and
 *     infeasible utterances are exact zeros, rows a missing forward call leaves are NaN;
 *   - the opt-in one-kernel path ("meet" option) is fp32-only: bf16 calls take the two-kernel path.
 * Any other logits_dtype (fp16 included) is CTCB_INVALID_VALUE.  The host entries, ctcb_pipe_*, ctcb_loss_grad_timed and
 * ctcb_proj_* are fp32-only.  A binding detects the feature by looking these symbols up. */
int ctcb_loss_grad_typed(const ctcb_problem_t* p, int32_t logits_dtype, void* workspace, size_t workspace_bytes,
                         void* stream);
int ctcb_forward_typed(const ctcb_problem_t* p, int32_t logits_dtype, int32_t keep_for_backward, void* workspace,
                       size_t workspace_bytes, void* stream);
int ctcb_backward_typed(const ctcb_problem_t* p, int32_t logits_dtype, void* workspace, size_t workspace_bytes,
                        void* stream);

/* Measurement aid (bench.py's roofline leg): ctcb_loss_grad with a CUDA event recorded on
 * `stream` after every kernel; synchronises and returns the per-kernel device times in launch
 * order (k_emit, k_walk, k_grad).  kernel_ms must hold 8 floats. */
int ctcb_loss_grad_timed(const ctcb_problem_t* p, void* workspace, size_t workspace_bytes,
                         void* stream, float* kernel_ms, int32_t* n_kernels);

/* Same operator with HOST buffers (what a `ctx=mx.cpu()` caller of the reference holds):
 * copies inputs host->device, runs ctcb_loss_grad, copies loss (and grad) back and
 * synchronises.  Device scratch is cached per device and grown on demand.  Used by
 * bench.py's end-to-end leg. */
int ctcb_loss_grad_host(const ctcb_problem_t* p, int device);

/* The training-step form of the host entry: inputs come from host buffers, the loss goes back to
 * the host, and the gradient STAYS on the device, where the model's backward pass consumes it
 * (train_ctc_ce.py:363-366: only `loss.asscalar()` crosses back).  *dev_grad receives the device
 * address of the gradient (same layout as the logits; library scratch, valid until the next
 * host-entry call on this device); p->grad is ignored. */
int ctcb_loss_grad_host_resident(const ctcb_problem_t* p, int device, float** dev_grad);

/* The host entry for a loop that prefetches (the reference's DataLoader hands the training loop the
 * next collated batch while the current one is in flight: train_ctc_ce.py:348-355 over
 * gluon DataLoader workers, batchify.py:51 shared-memory collation).  A pipe owns `depth` slots of
 * device buffers, a copy stream and a compute stream on `device`:
 *   ctcb_pipe_submit  enqueues host->device copies of the problem's inputs on the copy stream, the
 *                     kernels and the loss (loss_sum, status) device->host copies on the compute
 *                     stream, and returns a ticket WITHOUT waiting: the next batch's copy overlaps
 *                     this batch's kernels.  All pointers of `host_problem` are HOST pointers (page-
 *                     locked for the copies to be asynchronous); they must stay valid and untouched
 *                     until ctcb_pipe_wait(ticket) returns.  p->grad is ignored.  Inputs that lie in
 *                     ONE host allocation (checked with the driver: cuPointerGetAttribute range
 *                     queries, once per arena) with gaps < 4 KB move in one copy; separately
 *                     allocated arrays are copied one by one, whatever their addresses.  Submitting
 *                     when all slots hold uncollected batches first waits for the oldest.
 *   ctcb_pipe_wait    blocks until the ticket's batch is complete: the loss is in host_problem->loss,
 *                     *dev_grad (optional) is the device address of its gradient, in the logits'
 *                     layout, valid until `depth` more batches have been submitted.
 * One thread at a time per pipe.  Results are bit-identical to ctcb_loss_grad_host_resident. */
typedef struct ctcb_pipe ctcb_pipe_t;
int ctcb_pipe_create(int device, int depth, ctcb_pipe_t** out);
int ctcb_pipe_submit(ctcb_pipe_t* pipe, const ctcb_problem_t* host_problem, int64_t* ticket);
int ctcb_pipe_wait(ctcb_pipe_t* pipe, int64_t ticket, float** dev_grad);
int ctcb_pipe_destroy(ctcb_pipe_t* pipe);
/* bytes the last ctcb_pipe_submit moved host -> device.  *pulled is always 0 (the library always copies:
 * a kernel that pulled only the valid frames over PCIe was measured slower than the copy engine in
 * round 1 and removed; the argument stays for ABI stability). */
int ctcb_pipe_last_h2d_bytes(ctcb_pipe_t* pipe, int64_t* bytes, int32_t* pulled);

/* The operator's Backward for a caller that ran ctcb_loss_grad with head_grad = NULL in its
 * Forward (what MXNet's operator does: Forward stores the gradient, Backward multiplies it by
 * the head gradient -- SURVEY 8a row a8): grad[b, t, :] *= head_grad[b], in place. */
int ctcb_scale_rows(float* grad, int64_t stride_t, int64_t stride_b, int32_t T, int32_t B, int32_t V,
                    const float* head_grad, void* stream);

/* Greedy CTC decode of train_ctc_ce.py:149-160 / decode_ctc.py:123-143 (next-row scope,
 * SURVEY 8f rank 2): per utterance argmax over V for t < length, collapse repeats, drop
 * `blank`.  out_tokens (B, T) int32 (prefix valid), out_lengths (B,) int32.  Device buffers. */
int ctcb_greedy_decode(const float* logits, int64_t stride_t, int64_t stride_b,
                       const void* data_lengths, int32_t data_lengths_dtype,
                       int32_t T, int32_t B, int32_t V, int32_t blank,
                       int32_t* out_tokens, int32_t* out_lengths, void* stream);
/* The same with decode_ctc.py:120-140's <unk> rule: when the best symbol of a frame is `unk` the frame's
 * symbol is the SECOND best one (ties: lowest index); it is kept when it differs from the raw best symbol
 * of the previous frame -- the reference compares with trans[j-1], not with the substituted symbol -- and
 * is not the blank.  unk = -1: no rule (identical to ctcb_greedy_decode). */
int ctcb_greedy_decode_unk(const float* logits, int64_t stride_t, int64_t stride_b,
                           const void* data_lengths, int32_t data_lengths_dtype,
                           int32_t T, int32_t B, int32_t V, int32_t blank, int32_t unk,
                           int32_t* out_tokens, int32_t* out_lengths, void* stream);
/* ctcb_greedy_decode_unk for logits of type logits_dtype (CTCB_F32 or CTCB_BF16; bf16 values are compared after an exact
 * widening, ties -- frequent in bf16 -- still go to the lowest index). */
int ctcb_greedy_decode_typed(const void* logits, int32_t logits_dtype, int64_t stride_t, int64_t stride_b,
                             const void* data_lengths, int32_t data_lengths_dtype,
                             int32_t T, int32_t B, int32_t V, int32_t blank, int32_t unk,
                             int32_t* out_tokens, int32_t* out_lengths, void* stream);

/* Edit distance of each (reference, hypothesis) token pair of a batch: scripts/swbd/wer.py:45-68
 * (`_edit_distance`; next-row scope, SURVEY 8f rank 4).  ref (B, max_ref) / hyp (B, max_hyp)
 * int32 rows with the given row strides (elements) and lengths; `ctcb_greedy_decode`'s
 * out_tokens / out_lengths can be passed as hyp / hyp_len directly, so validation WER
 * (train_ctc_ce.py:149-168) needs no per-token host work.  out_dist (B,) int32.  When `totals` is
 * not NULL, totals[0] += sum of distances and totals[1] += sum of reference lengths: the two
 * numbers `compute_wer` (wer.py:9-43) divides.  Device buffers. */
int ctcb_edit_distance(const int32_t* ref, int64_t ref_stride, const int32_t* ref_len,
                       const int32_t* hyp, int64_t hyp_stride, const int32_t* hyp_len,
                       int32_t B, int32_t max_ref, int32_t max_hyp,
                       int32_t* out_dist, long long* totals, void* stream);

/* Sum of `count` doubles across the ranks of an NCCL communicator, in place, on `stream`
 * (ncclAllReduce, ncclSum).  NCCL is resolved with dlopen at first use, so libctcb.so has
 * no link-time NCCL dependency.  Replaces the host-side `+=` of `.asscalar()` values
 * (train_ctc_ce.py:367-368). */
int ctcb_loss_sum_allreduce(void* nccl_comm, double* dev_values, int32_t count, void* stream);

/* The same sum WITHOUT a collective kernel on the step's path: a mailbox per rank in device memory,
 * mapped into every peer process (CUDA IPC; the stores travel over NVLink / NVSwitch peer access).
 *   ctcb_mailbox_create    allocates this rank's mailbox on `device` (world <= 16).  `lag` (1..8, the same
 *                          on every rank) is the slack between the ranks in exchanges: an exchange
 *                          returns the sums handed over `lag` exchanges earlier
 *   ctcb_mailbox_handle    64-byte handle of the local mailbox; the caller gathers the handles of all
 *                          ranks in rank order (torch.distributed all_gather, MPI, a file ...)
 *   ctcb_mailbox_connect   maps the peers' mailboxes (handles: world x 64 bytes, rank order)
 *   ctcb_mailbox_exchange  one tiny kernel on `stream`: writes into dev_out[0..count) the all-rank sum
 *                          of the values handed to the exchange `lag` calls earlier (zeros before), then
 *                          stores dev_values[0..count) into every rank's mailbox and zeroes them
 *                          (count <= 6 doubles, e.g. loss sum, frames, utterances).  Every rank adds
 *                          the rows in rank order: identical bits everywhere.  Ranks need not meet:
 *                          a rank only waits for what its peers stored `lag` exchanges earlier.  All
 *                          ranks must issue the same number of exchanges.
 *   ctcb_mailbox_exchange_with_next   the same exchange as part of the next ctcb_loss_grad /
 *                          ctcb_forward / ctcb_backward this thread enqueues: the exchange kernel is
 *                          launched behind that call's gradient kernel as its programmatic dependent
 *                          and works beside the gradient kernel's last wave (ahead of the recursion
 *                          kernel, which then starts at once, on a forward-only call), so it is off
 *                          the step's path.  dev_values must not be the loss_sum that step
 *                          accumulates into: hand over the PREVIOUS step's partial sums (two
 *                          alternating slots).  Counts as one exchange.
 *   ctcb_mailbox_flush     dev_out = the all-rank sum of the LAST exchange's values (end of an epoch)
 * Replaces the host-side `+=` of `.asscalar()` values (train_ctc_ce.py:367-368) like
 * ctcb_loss_sum_allreduce does; bench.py --gpus N measures both (DESIGN.md section 8). */
typedef struct ctcb_mailbox ctcb_mailbox_t;
int ctcb_mailbox_create(int device, int rank, int world, int lag, ctcb_mailbox_t** out);
int ctcb_mailbox_handle(ctcb_mailbox_t* mailbox, void* handle64);
int ctcb_mailbox_connect(ctcb_mailbox_t* mailbox, const void* handles);
int ctcb_mailbox_exchange(ctcb_mailbox_t* mailbox, double* dev_values, int32_t count, double* dev_out, void* stream);
int ctcb_mailbox_exchange_with_next(ctcb_mailbox_t* mailbox, double* dev_values, int32_t count, double* dev_out);
int ctcb_mailbox_flush(ctcb_mailbox_t* mailbox, int32_t count, double* dev_out, void* stream);
int ctcb_mailbox_destroy(ctcb_mailbox_t* mailbox);

/* Introspection for tests/bench: number of kernel launches the last ctcb_loss_grad on this
 * thread enqueued, and the walker configuration it chose. */
int ctcb_last_launch_count(void);
int ctcb_last_walk_config(int32_t* pairs_per_lane, int32_t* warps);
/* Which gradient kernel the last call on this thread launched: 0 none, 1 k_grad (per-frame normalisation),
 * 2 k_grad2 (normalised by P(l|x); small vocabularies, from 64 utterances on), 3 k_meet (one-kernel path, opt-in). */
int ctcb_last_grad_kernel(void);

/* Tuning / experiment switches (tests and A/B measurements; a training loop never needs them).  Each
 * is read ONCE from the environment (CTCB_<NAME>, upper case) when the library is first used and can be
 * changed here; -1 = automatic.  Names: "walk_p", "walk_nw" (state pairs per lane / walker warps),
 * "walk_stages" (emission ring depth), "overlap" (gradient
 * kernel concurrent with the recursion kernel: 0/1), "fused" (0: always the k_emit path), "walk_per_sm",
 * "emit_staged", "grad_staged" (0: register variants for wide vocabularies), "grad2" (0/1: the gradient kernel
 * that normalises by P(l|x); automatic = from 64 utterances on), "grad2_blocks" (frame blocks per CTA of that
 * kernel), "meet" (1: the experimental one-kernel path of ctcb_meet.cuh), "meet_fwd" (loss evaluation without a
 * gradient: the alpha and the beta walker take half of the frames each and meet in the middle; automatic = while the
 * batch's walker CTAs are resident together), "proj_ctas" (fused projection: 2 = CTA pairs, 1 = single CTAs),
 * "proj_overlap" (0: the walkers run after the projection kernel instead of beside it), "proj_dbg" (measurement only),
 * "walk_pdl" (0: the recursion kernel is an ordinary launch instead of a programmatic one that waits on entry),
 * "grad_poll_ns" (back-off, in ns, between a gradient CTA's polls of the walkers' progress words; automatic = 128 / 256,
 * 1024 on the wide-vocabulary path).
 * walk_p / walk_nw / fused are part of the workspace layout: do not change them between ctcb_forward and ctcb_backward. */
int ctcb_set_option(const char* name, int32_t value);
int ctcb_get_option(const char* name, int32_t* value);

/* ---- output projection fused with the loss (SURVEY section 8f rank 1) ------------------------------------------------
 * Replaces the pair  `self.tgt_proj(net_out)`  (scripts/swbd/model.py:394-398 `nn.Dense(units=V, flatten=False)`, called
 * at model.py:424)  ->  `loss_function(out, ...)`  (train_ctc_ce.py:363 / :143) for vocabularies wider than 64 symbols:
 * logits[b,t,:] = hidden[b,t,:] . weight^T + bias is formed on the tensor cores (tcgen05, tf32 inputs read straight
 * from the fp32 tensors, fp32 accumulation in tensor memory) and reduced to what the lattice recursion reads -- row
 * maximum, softmax normaliser, the utterance's own label columns -- before it leaves the SM (csrc/ctcb_proj.cuh).
 * All pointers are device pointers.  hidden: (B, T, K) in any T/B strides (elements), unit stride along K; weight: (V, K)
 * row-major, gluon's Dense layout (units, in_units); strides and K multiples of 16 bytes, 16-byte aligned bases.
 * operand_dtype CTCB_PROJ_F32: fp32 tensors, tf32 product; CTCB_PROJ_BF16: bfloat16 tensors (mixed-precision encoders),
 * exact products at twice the tensor rate.  Accumulation, bias, logits and everything behind them are fp32 either way. */
#define CTCB_PROJ_F32 0
#define CTCB_PROJ_BF16 1
typedef struct ctcb_proj {
    const void* hidden;
    int64_t hidden_stride_t, hidden_stride_b;
    int32_t K;
    const void* weight;
    const float* bias;              /* (V,) fp32 or NULL (Dense(use_bias=False)) */
    int32_t operand_dtype;          /* CTCB_PROJ_F32 / CTCB_PROJ_BF16: element type of hidden and weight */
} ctcb_proj_t;

/* Loss of one batch from the encoder output.  p->logits is an OUTPUT here: NULL = the logits are never stored (the
 * validation pass, train_ctc_ce.py:143); otherwise the (T,B,V) buffer (p->logits_stride_*) the projection is written to,
 * once, for the gradient kernel.  keep_for_backward as in ctcb_forward: with it (and p->logits) a following
 * ctcb_backward(p, ...) writes d loss / d logits into p->grad, from which d hidden = G . weight, d weight = G^T . hidden
 * and d bias = sum G are plain library GEMMs (gluon_e2e_asr_b200/proj.py).  keep_for_backward with p->logits = NULL: no
 * logits are stored, the gradient comes from ctcb_proj_backward (below).  p->logits_row_offsets is not supported.
 * CTCB_UNSUPPORTED for V <= 64 or V <= Lmax + 1 (there the logits are a few per cent of the projection's traffic and the
 * walkers' fused producers read them once anyway) and for label rows too long for the kernel's shared memory. */
int ctcb_proj_forward(const ctcb_proj_t* proj, const ctcb_problem_t* p, int32_t keep_for_backward, void* workspace,
                      size_t workspace_bytes, void* stream);
/* ctcb_proj_forward plus the greedy decode of ctcb_greedy_decode_unk on the logits the projection forms
 * (train_ctc_ce.py:143-160): blank = p->blank, frame counts = p->data_lengths (clamped like the parameter layer),
 * unk = -1 for no <unk> rule.  out_tokens (B, T) int32, hypothesis prefix then zeros; out_lengths (B,) int32.  Tokens and
 * lengths are those of ctcb_greedy_decode_unk on the logits the projection writes with keep_for_backward = 1 (bit for bit:
 * the epilogue compares the values it would store, in the same order).  Device buffers; out_tokens also serves as the
 * per-frame scratch between the projection and the collapse kernel.  CTCB_UNSUPPORTED for T too long for the collapse
 * kernel's shared memory (2 T ints <= 200 KB).  Detected by symbol, like the *_typed entries. */
int ctcb_proj_forward_decode(const ctcb_proj_t* proj, const ctcb_problem_t* p, int32_t keep_for_backward, int32_t unk,
                             int32_t* out_tokens, int32_t* out_lengths, void* workspace, size_t workspace_bytes,
                             void* stream);
/* Greedy decode from the encoder output WITHOUT labels (decode_ctc.py:118-140: `tgt_proj`, then the argmax with the <unk>
 * rule): ctcb_greedy_decode_typed's arguments with the projection in place of the logits.  The projection's epilogue keeps
 * each frame's best and second best symbol of the logits it forms, a second kernel collapses repeats and blanks; the logits
 * never reach HBM, no workspace, 2 launches.  Frame counts = data_lengths (data_lengths_dtype; truncated and clamped to
 * [0, T]) or T when NULL; unk = -1 (or below) for no <unk> rule.  out_tokens (B, T) int32, hypothesis prefix then zeros;
 * out_lengths (B,) int32.  Tokens and lengths are bit-identical to ctcb_proj_forward_decode's for the same projection,
 * lengths, blank and unk, whatever its labels (the same tiles in the same K order), hence to ctcb_greedy_decode_unk on the
 * logits ctcb_proj_forward stores.  Any V >= 1: no V > 64 / Lmax restriction (there is no lattice).  Device buffers;
 * CTCB_UNSUPPORTED for T too long for the collapse kernel (2 T ints <= 200 KB).  Detected by symbol. */
int ctcb_proj_greedy_decode(const ctcb_proj_t* proj, int32_t T, int32_t B, int32_t V,
                            const void* data_lengths, int32_t data_lengths_dtype,
                            int32_t blank, int32_t unk, int32_t* out_tokens, int32_t* out_lengths, void* stream);
/* ctcb_proj_forward(keep_for_backward=1) followed by ctcb_backward in one call: loss, p->logits and p->grad. */
int ctcb_proj_loss_grad(const ctcb_proj_t* proj, const ctcb_problem_t* p, void* workspace, size_t workspace_bytes,
                        void* stream);
/* The training call without the logits: ctcb_proj_forward(keep_for_backward=1) with p->logits = NULL keeps the walkers'
 * history and turns it into a table of normalised lattice occupancies in the workspace (one more launch, no logits
 * written); this entry then forms the product again on the tensor cores, tile by tile, and writes
 * p->grad = head_grad[b] * (softmax(logits) - occupancy) -- d loss / d logits, fp32, (B,T,V) in p->grad_stride_* -- without
 * the logits ever reaching HBM.  Same proj and problem as the forward (the same workspace, need_grad = 1 size of
 * ctcb_workspace_bytes); p->logits is ignored, p->head_grad NULL = 1.  Padded frames and infeasible utterances get zero
 * rows; a workspace that no such forward filled gets NaN rows (no wait, no hang).  Validation as ctcb_proj_loss_grad;
 * CTCB_UNSUPPORTED where ctcb_proj_forward is (V <= 64, V <= Lmax + 1, label rows too long for shared memory).  Detected
 * by symbol, like the *_typed entries. */
int ctcb_proj_backward(const ctcb_proj_t* proj, const ctcb_problem_t* p, void* workspace, size_t workspace_bytes,
                       void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CTCB_H_ */
