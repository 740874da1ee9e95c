"""Mean-field DCA contacts and sequence weights of an alignment, from every record and column of it, with no model::

    python -m rnamsm_b200.dca --MSA_file X.a2m_msa2 --out contacts.npy \
        [--theta 0.8] [--pseudocount 0.5] [--weights_out w.npy]

Saves the ``(L, L)`` float32 contact map and, with ``--weights_out``, the float64 ``(N,)`` sequence weights, and prints
N, L and Neff (the effective number of sequences at identity ``theta``).  See ``rnamsm_b200.coevolution``.
"""
from __future__ import annotations

import argparse
import sys

import numpy as np


def parse_args(argv=None) -> argparse.Namespace:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--MSA_file", required=True)
    ap.add_argument("--out", required=True, help=".npy of the (L, L) float32 contact map")
    ap.add_argument("--theta", type=float, default=0.8, help="identity threshold of the sequence weights, in (0, 1]")
    ap.add_argument("--pseudocount", type=float, default=0.5, help="pseudocount weight, in (0, 1)")
    ap.add_argument("--weights_out", default=None, help="optional .npy of the (N,) float64 sequence weights")
    ap.add_argument("--device", default="cuda")
    return ap.parse_args(argv)


def main(argv=None):
    a = parse_args(argv)
    from .alphabet import Alphabet, Vocab
    from .coevolution import dca_contacts
    from .ingest import ingest_msa
    tokens, _ = ingest_msa(a.MSA_file, Vocab(Alphabet()), sys.maxsize, sys.maxsize, "first", device=a.device)
    out = dca_contacts(tokens, theta=a.theta, pseudocount=a.pseudocount)
    np.save(a.out, out["contacts"].cpu().numpy())
    if a.weights_out:
        np.save(a.weights_out, out["weights"].cpu().numpy())
    N, C = tokens.shape
    print(f"N {N}  L {C - 1}  Neff {out['neff']:.2f} (theta {a.theta})  contacts -> {a.out}")


if __name__ == "__main__":
    main()
