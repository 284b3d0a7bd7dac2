"""B200-native CTC loss-and-gradient engine: drop-in for the ``warpctc_pytorch`` path of
carolinebear/pytorch_end2end_speech_recognition (see DESIGN.md, INTEGRATION.md)."""

from ._lib import B200CTCError  # noqa: F401
from .ctc import (CTCLoss, _CTC, concatenate_labels, cpu_ctc, ctc_loss, ctc_loss_and_grad,  # noqa: F401
                  ctc_loss_from_padded, gpu_ctc, workspace_bytes)
from .decode import BeamSearchDecoder, GreedyDecoder, beam_search_decode, greedy_decode  # noqa: F401
from .evaluation import compute_wer, edit_distance, evaluate_batch, posteriors, word_errors  # noqa: F401
from .lm import NGramLM  # noqa: F401
from .shard import allreduce_loss, balance_shards, shard_batch, sharded_ctc_loss  # noqa: F401

__version__ = "0.2.0"
