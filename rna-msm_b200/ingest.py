"""MSA ingest on the GPU (SURVEY.md section 8f row 1): ``.a2m_msa2`` file -> cleaned character matrix ->
(optional) diversity sub-sampling -> int64 token grid on the device, ready for ``MSATransformer.forward``.

Mirrors ``dataset.A2MDataset`` / ``RNADataset.__getitem__`` (dataset.py:79-125): ``MSA.from_fasta``
(utils/align.py:292-317), ``select_diverse`` (utils/align.py:165-181) and ``Vocab.encode``
(utils/tokenization.py:107-129).  The host only splits the file into records; cleaning, selection and
tokenisation run in ``librnamsm_b200.so`` (csrc/ingest.cu), so a 10^5-row alignment never goes through
Python loops or the external ``hhfilter`` binary.

``sample_method``: "first" (keep the first ``max_seqs`` rows -- what the reference does with whatever
hhfilter returns beyond the limit, utils/align.py:172-173; the hhfilter binary itself is not reproduced),
"diversity-max" / "diversity-min" (``MSA.greedy_select``, bit-identical selections)."""
from __future__ import annotations

import ctypes as C
import re
from typing import List, Tuple

import numpy as np
import torch

from . import _lib as L
from .alphabet import Vocab


def split_records(path: str) -> Tuple[List[str], bytes, np.ndarray]:
    """FASTA-style file -> (headers, record bodies back to back, int64 offsets [N+1])."""
    headers: List[str] = []
    bodies: List[bytes] = []
    with open(path, "rb") as f:
        data = f.read()
    # a record starts at a '>' in the FIRST column of a line (Bio.SeqIO); a '>' inside a header ("a->b") is text.
    # SeqIO reads in text mode, where a lone '\r' ends a line too
    if b"\r>" in data:
        data = data.replace(b"\r>", b"\n>")
    for rec in (b"\n" + data).split(b"\n>")[1:]:            # anything before the first record is ignored
        nl = min((i for i in (rec.find(b"\n"), rec.find(b"\r")) if i >= 0), default=-1)
        headers.append(rec[:nl if nl >= 0 else len(rec)].decode(errors="replace").strip())
        bodies.append(rec[nl + 1:] if nl >= 0 else b"")
    offsets = np.zeros(len(bodies) + 1, dtype=np.int64)
    np.cumsum([len(b) for b in bodies], out=offsets[1:])
    return headers, b"".join(bodies), offsets


# blanks at the end of a line: SeqIO rstrip()s every line (str.isspace() over ASCII), so these go; inside a line only
# the spaces go (csrc/ingest.cu msa_clean_kernel)
_TRAILING_BLANKS = re.compile(rb"[\t\x0b\x0c\x1c-\x1f ]+(?=[\r\n]|\Z)")


def cleaned_length(body: bytes) -> int:
    """Length of one record after SeqIO's line handling and the from_fasta rules (host: the first record only, to
    size the matrix)."""
    body = _TRAILING_BLANKS.sub(b"", body)
    return sum(1 for ch in body if not (97 <= ch <= 122 or ch in b".*\n\r "))


@torch.no_grad()
def ingest_msa(path: str, vocab: Vocab, max_seqs: int = 512, max_seqlen: int = 1024, sample_method: str = "first",
               device: str = "cuda") -> Tuple[torch.Tensor, torch.Tensor]:
    """-> (tokens int64 [R, L+1] on ``device``, selected row indices int32 [R])."""
    if sample_method not in ("first", "diversity-max", "diversity-min"):
        raise ValueError(f"sample_method {sample_method!r}: expected 'first', 'diversity-max' or 'diversity-min' "
                         "(the reference's default 'hhfilter' shells out to an external binary)")
    headers, raw, offsets = split_records(path)
    N = len(headers)
    if N == 0:
        raise FileNotFoundError(f"no records in {path}")
    Lc = cleaned_length(raw[offsets[0]:offsets[1]])
    dev = torch.device(device)
    L.device_check(dev)
    with torch.cuda.device(dev):
        st = L.stream_ptr()
        raw_d = torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(dev)
        off_d = torch.from_numpy(offsets).to(dev)
        chars = torch.empty((N, Lc), dtype=torch.uint8, device=dev)
        bad = torch.zeros(1, dtype=torch.int32, device=dev)
        L.check(L.lib.rnamsm_msa_clean(L.ptr(raw_d), L.ptr(off_d), N, Lc, L.ptr(chars), L.ptr(bad), st), "msa_clean")
        b = int(bad.item())
        if b:
            raise AssertionError(f"Seqlen Mismatch! record {b - 1} of {path} does not clean to {Lc} characters")  # utils/align.py:28-30
        R = min(N, max_seqs)
        if sample_method == "first" or N <= max_seqs:
            rows = torch.arange(R, dtype=torch.int32, device=dev)
        else:
            rows = torch.empty(R, dtype=torch.int32, device=dev)
            ws = torch.empty(L.lib.rnamsm_msa_greedy_workspace(N, R), dtype=torch.uint8, device=dev)
            L.check(L.lib.rnamsm_msa_greedy_select(L.ptr(chars), N, Lc, R, int(sample_method == "diversity-max"), L.ptr(rows),
                                                   L.ptr(ws), st), "msa_greedy_select")
        lut = np.full(256, vocab.unk_idx, dtype=np.uint8)
        for tok, idx in vocab.alphabet.tok_to_idx.items():
            if len(tok) == 1:
                lut[ord(tok)] = idx
        lut_d = torch.from_numpy(lut).to(dev)
        Lt = min(Lc, max_seqlen - 1)                     # RandomCropDataset(max_seqlen) upper bound, dataset.py:142-158
        tokens = torch.empty((R, Lc + 1), dtype=torch.int64, device=dev)
        L.check(L.lib.rnamsm_msa_tokenize(L.ptr(chars), Lc, L.ptr(rows), R, L.ptr(lut_d), vocab.alphabet.tok_to_idx["<cls>"],
                                          L.ptr(tokens), st), "msa_tokenize")
        if Lt < Lc:
            tokens = tokens[:, :Lt + 1].contiguous()
    return tokens, rows
