"""rnamsm_b200 -- B200-native RNA-MSM MSA-transformer forward (emb + 120 tied-row attention maps).

Python host side of ``librnamsm_b200.so`` (C ABI in ``include/rnamsm_b200.h``); mirrors the
reference's ``MSATransformer`` / ``AxialTransformerLayer`` API.  Importing this package loads
the CUDA library and raises if it is missing -- there is no CPU or PyTorch fallback.
"""
from . import _lib  # noqa: F401  (loads librnamsm_b200.so, fails loudly when absent)
from .alphabet import Alphabet, Vocab, read_msa, tokenize_msa  # noqa: F401
from .model import MSATransformer, jacobian_entries, plan_score_group  # noqa: F401
from .mutations import parse_mutant  # noqa: F401
from .modules import (AxialTransformerLayer, ColumnSelfAttention, ContactPredictionHead,  # noqa: F401
                      FeedForwardNetwork, LearnedPositionalEmbedding, NormalizedResidualBlock, RobertaLMHead,
                      RowSelfAttention)
from .inference import (extract_features, extract_features_batch, extract_features_batch_streamed,  # noqa: F401
                        extract_features_streamed, extract_features_windowed, pack_rsa_input, pack_ss_input,
                        plan_batches, run_inference)
from .ingest import ingest_msa  # noqa: F401
from .coevolution import dca_contacts, sequence_weights  # noqa: F401
from .structure import dot_bracket, fold_pairs, write_bpseq, write_ct  # noqa: F401

__all__ = ["MSATransformer", "AxialTransformerLayer", "RowSelfAttention", "ColumnSelfAttention",
           "FeedForwardNetwork", "NormalizedResidualBlock", "LearnedPositionalEmbedding", "RobertaLMHead",
           "ContactPredictionHead", "Alphabet", "Vocab", "read_msa", "tokenize_msa", "extract_features",
           "run_inference", "ingest_msa", "pack_ss_input", "extract_features_streamed", "extract_features_batch",
           "extract_features_batch_streamed", "pack_rsa_input", "plan_batches", "plan_score_group", "parse_mutant",
           "jacobian_entries", "extract_features_windowed", "sequence_weights", "dca_contacts", "fold_pairs", "dot_bracket",
           "write_ct", "write_bpseq"]
