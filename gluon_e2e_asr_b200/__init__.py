"""gluon_e2e_asr_b200 -- the CTC training-loss path of Hex-Lee/gluon-e2e-asr, rebuilt for B200.

Scope is ONE path (SURVEY.md section 8): ``CtcLoss`` / ``ctc_loss`` forward+backward, the
batch sharding around it and the next rows: greedy CTC decode, the length-bucketing samplers and
pinned collation that feed it, and the edit distance behind the validation WER.  Everything else the reference
contains is out of scope on purpose.
"""
from .loss import CtcLoss
from .batch import PinnedBatch
from .pipeline import HostPipeline
from .ops import CTCLoss, ctc_loss, ctc_loss_and_grad, edit_distance, greedy_decode, workspace_bytes
from .proj import ProjCtcLoss, proj_ctc_eval, proj_ctc_loss, proj_greedy_decode
from .sampler import FixedBucketSampler, SortedBucketSampler, SortedSampler
from .sharding import (PeerLossSum, balanced_assignment, loss_sum_allreduce, shard_for_rank,
                       split_and_load, split_slices)

__all__ = ["CtcLoss", "CTCLoss", "ctc_loss", "ctc_loss_and_grad", "greedy_decode",
           "workspace_bytes", "split_and_load", "split_slices", "balanced_assignment",
           "shard_for_rank", "loss_sum_allreduce", "PeerLossSum", "edit_distance", "PinnedBatch", "HostPipeline", "FixedBucketSampler",
           "SortedBucketSampler", "SortedSampler", "ProjCtcLoss", "proj_ctc_loss", "proj_ctc_eval", "proj_greedy_decode"]
