/* ctcb_dlpack.h -- DLPack hand-off for libctcb.so.
 *
 * The reference hands NDArrays to its operator; a Python caller of this library hands
 * DLPack capsules (torch.utils.dlpack.to_dlpack / mx.nd.NDArray.to_dlpack_for_read).  The
 * struct definitions below restate the public DLPack ABI (dlpack.h, v0.x `DLManagedTensor`
 * layout, which v1.x keeps as the legacy struct) so the library needs no external header.
 *
 * Ownership: the library BORROWS each DLManagedTensor for the duration of the call.  It
 * never calls `deleter`, never renames the capsule and keeps no pointer after returning
 * (the enqueued kernels keep using the device memory: the caller keeps the tensors alive
 * until the stream has run, as with any async CUDA op).
 */
#ifndef CTCB_DLPACK_H_
#define CTCB_DLPACK_H_

#include <stdint.h>
#include "ctcb.h"

#ifdef __cplusplus
extern "C" {
#endif

#ifndef DLPACK_DLPACK_H_   /* do not clash with a real dlpack.h */
typedef enum { kDLCPU = 1, kDLCUDA = 2, kDLCUDAHost = 3, kDLCUDAManaged = 13 } DLDeviceType;
typedef struct { int32_t device_type; int32_t device_id; } DLDevice;
typedef enum { kDLInt = 0U, kDLUInt = 1U, kDLFloat = 2U, kDLBfloat = 4U } DLDataTypeCode;
typedef struct { uint8_t code; uint8_t bits; uint16_t lanes; } DLDataType;
typedef struct {
    void* data;
    DLDevice device;
    int32_t ndim;
    DLDataType dtype;
    int64_t* shape;
    int64_t* strides;      /* in elements; NULL = compact row-major */
    uint64_t byte_offset;
} DLTensor;
typedef struct DLManagedTensor {
    DLTensor dl_tensor;
    void* manager_ctx;
    void (*deleter)(struct DLManagedTensor* self);
} DLManagedTensor;
#endif

/* layout flags for ctcb_loss_grad_dlpack */
#define CTCB_LAYOUT_TNC   0   /* logits/grad are (T,B,V): the operator's layout            */
#define CTCB_LAYOUT_NTC   1   /* logits/grad are (B,T,V): CtcLoss(layout='NTC'), loss.py:123 */
#define CTCB_LABEL_TN     2   /* labels are (Lmax,B): CtcLoss(label_layout='TN'), loss.py:125 */
#define CTCB_KEEP_FOR_BACKWARD 4   /* with CTCB_PHASE_FORWARD: keep the history for a later backward */
#define CTCB_PHASE_FUSED     (0 << 8)   /* ctcb_loss_grad  */
#define CTCB_PHASE_FORWARD   (1 << 8)   /* ctcb_forward    */
#define CTCB_PHASE_BACKWARD  (2 << 8)   /* ctcb_backward   */

/* mx.nd.contrib.ctc_loss(data, label, data_lengths, label_lengths, use_data_lengths,
 * use_label_lengths, blank_label) (loss.py:134-139) on DLPack tensors.
 *   logits        fp32 or bfloat16 CUDA, 3-d, unit stride on the last axis, any T/B strides (bf16: ctcb.h, *_typed)
 *   labels        2-d, int32/int64/float32/float64, CUDA
 *   data_lengths  1-d (B,) or NULL  == use_data_lengths=False
 *   label_lengths 1-d (B,) or NULL  == use_label_lengths=False
 *   head_grad     1-d (B,) fp32 or NULL (= ones)
 *   loss          1-d (B,) fp32, written
 *   grad          same shape and dtype as logits, written; NULL = forward only
 *   loss_sum      0/1-d float64 scalar accumulated in place, or NULL
 *   blank_last    0: blank_label='first' (the reference, loss.py:139), 1: 'last'
 */
int ctcb_loss_grad_dlpack(const DLManagedTensor* logits, const DLManagedTensor* labels,
                          const DLManagedTensor* data_lengths,
                          const DLManagedTensor* label_lengths,
                          const DLManagedTensor* head_grad, DLManagedTensor* loss,
                          DLManagedTensor* grad, DLManagedTensor* loss_sum,
                          int32_t blank_last, int32_t layout_flags, void* workspace,
                          size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CTCB_DLPACK_H_ */
