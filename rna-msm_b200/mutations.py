"""Mutant strings for LM-head scoring (``MSATransformer.score_mutations``, ``python -m rnamsm_b200.score``).

A mutant is one or more substitutions joined by ``:``, each ``<wt><index><mt>`` such as ``"G12A"`` or
``"G12A:C30U"``.  Indices are 1-based residues of the query row, so residue ``k`` is token-grid column ``k`` (column 0
holds ``<cls>``).  Letters are the alphabet's standard tokens (``A G C U X N -``); ``T`` is read as ``U``, as the MSA
readers clean it.  Host-only: nothing here touches the GPU.
"""
from __future__ import annotations

import re
from typing import List, Sequence, Tuple

_SUB = re.compile(r"^([A-Za-z-])(\d+)([A-Za-z-])$")


def letter_index(letter: str, vocab) -> int:
    """Token index of one standard letter (``T`` -> ``U``); ``ValueError`` for anything else."""
    ch = "U" if letter == "T" else letter
    if ch not in vocab.alphabet.standard_toks:
        raise ValueError(f"unknown residue letter {letter!r} (expected one of {''.join(vocab.alphabet.standard_toks)} or T)")
    return vocab.tokens_to_idx[ch]


def parse_mutant(spec: str, query: Sequence[int], vocab) -> List[Tuple[int, int, int]]:
    """``"G12A:C30U"`` -> ``[(column, wt_token, mt_token), ...]`` checked against ``query``, the token ids of the
    scored row (``[C]``, column 0 = ``<cls>``).  ``ValueError`` when a substitution is malformed, names an unknown
    letter, an index outside ``1 .. C-1`` or a ``<pad>`` column, a wild type that is not the query's token there, or
    the same position twice."""
    subs = spec.strip().split(":")
    if not spec.strip():
        raise ValueError("empty mutant")
    out, seen = [], set()
    for s in subs:
        m = _SUB.match(s.strip())
        if m is None:
            raise ValueError(f"mutant {spec!r}: {s!r} is not <wt><index><mt>, e.g. G12A")
        wt, mt = letter_index(m.group(1), vocab), letter_index(m.group(3), vocab)
        col = int(m.group(2))
        if not 1 <= col < len(query):
            raise ValueError(f"mutant {spec!r}: index {col} outside residues 1..{len(query) - 1}")
        if int(query[col]) == vocab.pad_idx:
            raise ValueError(f"mutant {spec!r}: index {col} is a padding column of the query")
        if int(query[col]) != wt:
            have = vocab.tokens[int(query[col])]
            raise ValueError(f"mutant {spec!r}: wild type {m.group(1)!r} at {col} but the query has {have!r}")
        if col in seen:
            raise ValueError(f"mutant {spec!r}: position {col} appears twice")
        seen.add(col)
        out.append((col, wt, mt))
    return out


def read_mutants(path: str) -> List[str]:
    """One mutant per line; blank lines and ``#`` comments are skipped."""
    with open(path) as f:
        return [ln.strip() for ln in f if ln.strip() and not ln.lstrip().startswith("#")]
