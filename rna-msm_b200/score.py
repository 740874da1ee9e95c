"""Zero-shot mutant scoring with the LM head (the scoring half of the reference's ``utils/likelihood.py``)::

    python -m rnamsm_b200.score --MSA_file X.a2m_msa2 --mutations muts.txt --out scores.tsv \
        [--method masked-marginals|wt-marginals] [--marginals_out marginals.npy]

The alignment is read like ``rnamsm_b200.inference`` reads it; its first row is the query.  ``muts.txt`` holds one
mutant per line (``G12A`` or ``G12A:C30U``, 1-based query residues).  Writes a TSV with columns ``mutant`` and
``score`` in input order and prints the query's pseudo-log-likelihood.  ``--marginals_out`` saves the log-probabilities
of every query residue ``[L, V]`` (float32) under the chosen method.
"""
from __future__ import annotations

import argparse
import math

import numpy as np

from .ingest import ingest_msa
from .inference import build_model
from .mutations import read_mutants


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--MSA_file", required=True)
    ap.add_argument("--mutations", required=True, help="one mutant per line")
    ap.add_argument("--out", required=True, help="TSV: mutant, score")
    ap.add_argument("--method", default="masked-marginals", choices=["masked-marginals", "wt-marginals"])
    ap.add_argument("--marginals_out", default=None, help="optional .npy of the query's [L, V] log-probabilities")
    ap.add_argument("--device", default="cuda")
    ap.add_argument("--model_path", default=None, help="Lightning checkpoint ('state_dict'); random init if omitted")
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16", "bf16_pure", "tf32x3", "fp32"])
    ap.add_argument("--max_seqs_per_msa", type=int, default=512)
    ap.add_argument("--sample_method", default="first", choices=["first", "diversity-max", "diversity-min"])
    ap.add_argument("--max_seqlen", type=int, default=1024)
    ap.add_argument("--no_embed_positions_msa", action="store_true")
    a = ap.parse_args(argv)
    model, vocab = build_model(a.model_path, a.device, a.precision, embed_positions_msa=not a.no_embed_positions_msa,
                               max_seqlen=a.max_seqlen)
    tokens, _ = ingest_msa(a.MSA_file, vocab, a.max_seqs_per_msa, a.max_seqlen, a.sample_method, device=str(model.device))
    mutants = read_mutants(a.mutations)
    scores = model.score_mutations(tokens, mutants, method=a.method)
    with open(a.out, "w") as f:
        f.write("mutant\tscore\n")
        for s, v in zip(mutants, scores.tolist()):
            f.write(f"{s}\t{v!r}\n")
    pll, per_position = model.pseudo_log_likelihood(tokens)
    L = per_position.numel()
    print(f"pseudo_log_likelihood\t{pll!r}\tpseudo_perplexity\t{math.exp(-pll / max(L, 1))!r}\tL\t{L}")
    if a.marginals_out:
        lp = model.masked_marginals(tokens, masked=a.method == "masked-marginals")
        np.save(a.marginals_out, lp.cpu().numpy())
    print(f"{len(mutants)} mutants scored -> {a.out}")


if __name__ == "__main__":
    main()
