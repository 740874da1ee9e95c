"""Contacts of an alignment's query read from the LM head alone, by the categorical Jacobian::

    python -m rnamsm_b200.jacobian --MSA_file X.a2m_msa2 --out contacts.npy \
        [--jacobian_out J.npy] [--alphabet AGCU] [--precision fp16]

The alignment is read like ``rnamsm_b200.score`` reads it; its first row is the query.  Every query residue is
substituted by every other letter of ``--alphabet`` and ``MSATransformer.categorical_jacobian`` records how the LM-head
logits of all residues move (about ``3L + 1`` forwards of the alignment for ``AGCU``).  Saves the ``(L, L)`` float32
contact map of the query's non-pad residues and, with ``--jacobian_out``, the Jacobian ``(L, A, L, A)`` float32.  No
contact regression is used, so a checkpoint without a fitted ``contact_head`` works too.
"""
from __future__ import annotations

import argparse

import numpy as np

from .ingest import ingest_msa
from .inference import build_model


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--MSA_file", required=True)
    ap.add_argument("--out", required=True, help=".npy of the (L, L) float32 contact map")
    ap.add_argument("--jacobian_out", default=None, help="optional .npy of the (L, A, L, A) float32 Jacobian")
    ap.add_argument("--alphabet", default="AGCU", help="substituted letters, distinct, from A G C U X N -")
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
    contacts, J = model.categorical_jacobian(tokens, alphabet=a.alphabet, return_jacobian=True)
    np.save(a.out, contacts.cpu().numpy())
    if a.jacobian_out:
        np.save(a.jacobian_out, J.cpu().numpy())
    print(f"contacts {tuple(contacts.shape)} -> {a.out}")


if __name__ == "__main__":
    main()
