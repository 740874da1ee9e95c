"""Secondary structure of an alignment's query (its first record), folded on the device from one of the library's pair
maps::

    python -m rnamsm_b200.fold --MSA_file X.a2m_msa2 --out_prefix P --source {contact-head,jacobian,dca,npy} \
        [--map m.npy] [--model_path ckpt] [--precision fp16] [--mode mea|score] [--gamma 1] [--threshold 0] \
        [--min_loop 3] [--no_canonical]

Sources: ``contact-head``, the contact head's pair probabilities (``forward_windows``, so any length; bit-identical
to ``forward`` up to 1023 residues); ``jacobian``, the categorical Jacobian's APC contacts; ``dca``, mean-field DCA
over every record of the file; ``npy``, an ``(L, L)`` map from ``--map``.  ``contact-head`` and ``npy`` fold with
``--mode mea`` by default, ``jacobian`` and ``dca`` with ``--mode score``.  Pairs are canonical (AU, GC, GU) unless
``--no_canonical``.  Writes ``P.ct``, ``P.bpseq`` and ``P.dbn``.  See ``rnamsm_b200.structure``.
"""
from __future__ import annotations

import argparse
import math
import os
import sys

import numpy as np

SOURCES = ("contact-head", "jacobian", "dca", "npy")
DEFAULT_MODE = {"contact-head": "mea", "npy": "mea", "jacobian": "score", "dca": "score"}


def parse_args(argv=None) -> argparse.Namespace:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--MSA_file", required=True)
    ap.add_argument("--out_prefix", required=True, help="writes <prefix>.ct, <prefix>.bpseq and <prefix>.dbn")
    ap.add_argument("--source", required=True, choices=SOURCES)
    ap.add_argument("--map", default=None, help="(L, L) .npy pair map of the query (--source npy only)")
    ap.add_argument("--model_path", default=None, help="Lightning checkpoint ('state_dict'); random init if omitted")
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16", "bf16_pure", "tf32x3", "fp32"])
    ap.add_argument("--max_seqs_per_msa", type=int, default=512, help="rows given to the model")
    ap.add_argument("--sample_method", default="first", choices=["first", "diversity-max", "diversity-min"])
    ap.add_argument("--mode", default=None, choices=["mea", "score"], help="default: by source")
    ap.add_argument("--gamma", type=float, default=1.0, help="pair weight of --mode mea, > 0")
    ap.add_argument("--threshold", type=float, default=0.0, help="pairs need a map value above it")
    ap.add_argument("--min_loop", type=int, default=3, help="pairs (i, j) need j - i > min_loop")
    ap.add_argument("--no_canonical", action="store_true", help="allow any letters to pair")
    ap.add_argument("--device", default="cuda")
    a = ap.parse_args(argv)
    if (a.source == "npy") != (a.map is not None):
        ap.error("--map is required with --source npy and only allowed there")
    if not (a.gamma > 0 and math.isfinite(a.gamma)):
        ap.error(f"--gamma {a.gamma} must be positive and finite")
    if not math.isfinite(a.threshold):
        ap.error(f"--threshold {a.threshold} must be finite")
    if a.min_loop < 0:
        ap.error(f"--min_loop {a.min_loop} must be >= 0")
    if a.mode is None:
        a.mode = DEFAULT_MODE[a.source]
    return a


def query_sequence(tokens, vocab) -> str:
    """Letters of row 0 after BOS; tokens outside A G C U X N - read as N."""
    letters = []
    for t in tokens[0, 1:].tolist():
        tok = vocab.tokens[t]
        letters.append(tok if tok in "AGCUXN-" and len(tok) == 1 else "N")
    return "".join(letters)


def pair_map(a, device):
    """-> (query tokens' letters, fp32 [L, L] map on the device, record 0's header)"""
    import torch

    from .alphabet import Alphabet, Vocab
    from .coevolution import dca_contacts
    from .inference import build_model
    from .ingest import ingest_msa, split_records

    name = split_records(a.MSA_file)[0][0] or os.path.basename(a.MSA_file)
    if a.source == "dca":
        vocab = Vocab(Alphabet())
        tokens, _ = ingest_msa(a.MSA_file, vocab, sys.maxsize, sys.maxsize, "first", device=device)
        return query_sequence(tokens, vocab), dca_contacts(tokens)["contacts"], name
    if a.source == "npy":
        vocab = Vocab(Alphabet())
        tokens, _ = ingest_msa(a.MSA_file, vocab, 1, sys.maxsize, "first", device=device)
        m = np.load(a.map)
        return query_sequence(tokens, vocab), torch.from_numpy(np.ascontiguousarray(m, dtype=np.float32)).to(device), name
    model, vocab = build_model(a.model_path, device, a.precision)
    tokens, _ = ingest_msa(a.MSA_file, vocab, a.max_seqs_per_msa, sys.maxsize, a.sample_method,
                           device=str(model.device))
    if a.source == "contact-head":
        contacts = model.forward_windows(tokens, return_contacts=True)["contacts"]
    else:
        contacts = model.categorical_jacobian(tokens)
    return query_sequence(tokens, vocab), contacts, name


def main(argv=None):
    a = parse_args(argv)
    from .structure import dot_bracket, fold_pairs, write_bpseq, write_ct

    seq, S, name = pair_map(a, a.device)
    if S.shape != (len(seq), len(seq)):
        raise ValueError(f"the map is {tuple(S.shape)} but the query has {len(seq)} residues")
    pairs, score = fold_pairs(S, seq, mode=a.mode, gamma=a.gamma, threshold=a.threshold, min_loop=a.min_loop,
                              canonical=not a.no_canonical)
    db = dot_bracket(pairs)
    write_ct(a.out_prefix + ".ct", name, seq, pairs)
    write_bpseq(a.out_prefix + ".bpseq", seq, pairs)
    with open(a.out_prefix + ".dbn", "w") as f:
        f.write(f">{name}\n{seq}\n{db}\n")
    print(f"L {len(seq)}  pairs {db.count('(')}  score {score:.6g} ({a.source}, {a.mode})  -> {a.out_prefix}"
          ".ct/.bpseq/.dbn")


if __name__ == "__main__":
    main()
