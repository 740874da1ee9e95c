"""Cases and exact references for the kernels in front of the model and behind it: the alignment ingest
(csrc/ingest.cu: msa_clean, greedy_select, tokenize) and the predictor-input packing (csrc/contact.cu: ss_pack,
rsa_pack).  Device-agnostic numpy; tests/test_ingest_cases_cpu.py proves that each case does what it claims and
tests/test_gpu_ingest_edges.py runs them through the C ABI.  Every output of these kernels is exact (row indices,
token ids, copied or z-scored floats), so every comparison is bit for bit.

* ``seqio_records``: the record splitting and line handling of Bio.SeqIO's FASTA parser, which ``MSA.from_fasta``
  iterates, followed by ``oracle/msa_ingest_ref.clean_sequence``: the reference for ``split_records`` + msa_clean.
* Alignment builders for greedy_select, each named for the launch branch of ingest.cu it reaches
  (``launch_geometry`` restates the launch formulas).
* ``kernel_sum_replay``: the kernel's ``np_pairwise_sum`` in float64, vectorised over rows, and its sequential variant;
  ``greedy_trace`` replays the whole selection with either, to show which cases separate the two summation orders.
* Messy FASTA writers, tokenizer inputs and the SS / RSA pack cases with their references.
"""
from __future__ import annotations

import io
from typing import List, NamedTuple, Tuple

import numpy as np

from oracle import msa_ingest_ref as I
from oracle import msa_ref as O

# ---------------------------------------------------------------------------------------------------- FASTA parsing

BLANKS = "\t\x0b\x0c\x1c\x1d\x1e\x1f"    # str.isspace() over ASCII, less ' ' and the line ends: what rstrip() removes


def seqio_records(data: bytes) -> List[Tuple[str, str]]:
    """``Bio.SeqIO.parse(path, "fasta")`` on an ASCII file: ``[(title, sequence)]``.

    SeqIO opens the path in text mode, so universal newlines apply: ``'\\r\\n'`` and a lone ``'\\r'`` end a line just
    like ``'\\n'``.  The parser is ``SimpleFastaParser`` (Biopython 1.79 - 1.84, ``Bio/SeqIO/FastaIO.py``), restated
    statement for statement:

        for line in handle:                          # text before the first record is skipped
            if line[0] == ">":
                title = line[1:].rstrip()
                break
        else:
            return
        lines = []
        for line in handle:
            if line[0] == ">":
                yield title, "".join(lines).replace(" ", "").replace("\\r", "")
                lines = []
                title = line[1:].rstrip()
                continue
            lines.append(line.rstrip())
        yield title, "".join(lines).replace(" ", "").replace("\\r", "")

    So a space is dropped anywhere, and every other blank (tab, '\\v', '\\f', '\\x1c' - '\\x1f') only at the end of a
    line: a tab inside a line survives into the sequence, a '\\v' or '\\f' at the end of a line does not."""
    handle = io.TextIOWrapper(io.BytesIO(data), encoding="ascii", newline=None)
    out = []
    for line in handle:
        if line[0] == ">":
            title = line[1:].rstrip()
            break
    else:
        return out
    lines = []
    for line in handle:
        if line[0] == ">":
            out.append((title, "".join(lines).replace(" ", "").replace("\r", "")))
            lines = []
            title = line[1:].rstrip()
            continue
        lines.append(line.rstrip())
    out.append((title, "".join(lines).replace(" ", "").replace("\r", "")))
    return out


def reference_rows(data: bytes) -> List[str]:
    """MSA.from_fasta's rows of a file: the SeqIO sequences through clean_sequence (utils/align.py:311-313)."""
    return [I.clean_sequence(s) for _, s in seqio_records(data)]


# ---------------------------------------------------------------------------------------------------- messy files

def _line_end(rng, style):
    if style == "mixed":
        return ["\n", "\r\n", "\r"][int(rng.integers(0, 3))]
    return {"lf": "\n", "crlf": "\r\n", "cr": "\r"}[style]


def write_messy(rows: List[str], rng, ends="lf", width=23, noise=True, trailing="", preamble="", header=">seq{n} a->b"):
    """Rows of a cleaned matrix back into a hostile a2m file whose from_fasta rows are ``rows`` again: lowercase and
    '.' insertions, T for U, IUPAC codes for X, spaces anywhere, ``trailing`` blanks before every line end, line ends
    ``ends`` ('lf', 'crlf', 'cr' or 'mixed'), lines wrapped at ``width`` but never after a blank or a space (a blank
    the row keeps would become trailing and go).  Extends ``_write_fasta`` of tests/test_ingest.py."""
    out = [preamble]
    for n, row in enumerate(rows):
        toks = []
        for ch in row:
            if noise and rng.random() < 0.15:
                toks.append(str(rng.choice(list("acgu."))) * int(rng.integers(1, 3)))
            if ch == "U" and noise and rng.random() < 0.5:
                ch = "T"
            elif ch == "X" and noise:
                ch = str(rng.choice(list("XNRYKMSWBDHV")))
            if noise and rng.random() < 0.1:
                toks.append(" ")
            toks.append(ch)
        out.append(header.format(n=n) + _line_end(rng, ends))
        line = ""
        for t in toks:
            line += t
            if len(line) >= width and not line[-1].isspace():
                out.append(line + trailing + _line_end(rng, ends))
                line = ""
        if line:
            out.append(line + trailing + _line_end(rng, ends))
    return "".join(out).encode("ascii")


def _rows(n, L, seed, alphabet="AGCU-X"):
    rng = np.random.default_rng(seed)
    return ["".join(rng.choice(list(alphabet), L)) for _ in range(n)]


def messy_files():
    """name -> (file bytes, well_formed).  A well-formed file cleans every record to the first record's length."""
    rng = np.random.default_rng(23)
    blank_rows = ["".join(r) for r in _rows(12, 40, 1, "AGCU-X\t\x0b\x0c\x1c\x1f")]
    blank_rows = [("A" + r[1:-1] + "G") for r in blank_rows]
    files = {
        "lf": (write_messy(_rows(40, 33, 2), rng), True),
        "crlf": (write_messy(_rows(40, 33, 3), rng, ends="crlf"), True),
        "cr": (write_messy(_rows(40, 33, 4), rng, ends="cr"), True),
        "mixed_ends": (write_messy(_rows(40, 65, 5), rng, ends="mixed", width=17), True),
        "midline_blanks": (write_messy(blank_rows, rng, width=9), True),
        "trailing_blanks": (write_messy(_rows(30, 50, 6), rng, ends="mixed", trailing=" \t\x0b\x0c\x1c\x1d\x1e\x1f\t"), True),
        "headers": (write_messy(_rows(20, 31, 7), rng, preamble="# made by hand\n\n  x>y\n;>z\n",
                                header=">h{n} >a->b\t|x>y \x0c"), True),
        "one_line": (write_messy(_rows(16, 200, 8), rng, width=10 ** 6, ends="crlf"), True),
    }
    # records cleaning to nothing, to too much and too little, next to well-formed ones
    rows = _rows(10, 20, 9)
    bad = write_messy(rows[:3], rng).decode() + ">empty\n>empty too\n\n \t\n" + \
        write_messy(rows[3:6], rng, header=">mid{n}").decode() + ">long\n" + rows[6] + "ACGUA\n" + \
        ">short\n" + rows[7][:-1] + "\t\n" + ">last\n" + rows[8]
    files["malformed"] = (bad.encode(), False)
    files["overlong_only"] = ((">a\nACGU\n>b\nACGUU\n>c\nAC\tGU\n>d\nACGU\n").encode(), False)
    files["chunk_edges"] = (chunk_edge_file(), True)
    return files


def chunk_edge_file():
    """Record bodies of 31 / 32 / 33 / 63 / 64 / 65 / 1023 / 1024 / 1025 bytes (the clean kernel reads 32 bytes per warp
    step), each with a blank run that straddles a 32-byte step and then meets either text (kept) or the end of the
    body (dropped), and 4 tabs inside a 74-byte blank run inside a line.  Every record cleans to 16 characters."""
    recs = []
    for B in (31, 32, 33, 63, 64, 65, 1023, 1024, 1025):
        # text, filler '.', then a blank run that ends the body (the end of its last line: dropped)
        recs.append("ACGUACGU" + "." * (B - 21) + "ACGUACGU" + " \t\x0b\x0c\t")
        # a run of 4 kept blanks and a space across the last 32-byte step before B - 11, then text
        at = max(6, 32 * ((B - 12) // 32) - 2)
        recs.append("ACGUAC" + "." * (at - 6) + "\t \x0b\x0c\x1c" + "ACGUAC" + "." * (B - at - 11))
    recs.append("AC" + "\t" * 4 + " " * 70 + "GUACGUACGU" + " \t\n \t\x0b")   # 4 tabs in a 74-byte blank run
    return "".join(f">r{n}\n{b}\n" for n, b in enumerate(recs)).encode("ascii")


# ---------------------------------------------------------------------------------------------------- greedy select

SM_SLOTS = 148 * 4        # ingest.cu: per-launch block cap of greedy_hamming_kernel / greedy_mean_kernel


def launch_geometry(N, L, num):
    """The launch formulas of rnamsm_msa_greedy_select (ingest.cu) and what they imply for one case."""
    blocks_h = min(-(-N // 8), SM_SLOTS)
    blocks_m = min(-(-N // 256), SM_SLOTS)
    return {
        "blocks_h": blocks_h, "hamming_sweeps": -(-N // (blocks_h * 8)),
        "blocks_m": blocks_m, "mean_sweeps": -(-N // (blocks_m * 256)),
        "pick_per_lane": -(-blocks_m // 32),
        "lut_bytes": (L + 1) * 8, "big_lut": (L + 1) * 8 > 48 * 1024,
        "max_k": num - 1, "recursion": num - 1 > 128, "sort_threads_used": num,
    }


def family(N, L, ancestors, rate, seed, alphabet="AGCU-"):
    """Rows derived from a few random ancestors by point mutation at ``rate``: many rows at equal mean distance from
    the picks, so exact ties (decided by float64 rounding) occur deep into the selection."""
    rng = np.random.default_rng(seed)
    a = np.frombuffer(alphabet.encode(), np.uint8)
    anc = a[rng.integers(0, len(a), (ancestors, L))]
    x = anc[rng.integers(0, ancestors, N)].copy()
    mut = rng.random((N, L)) < rate
    x[mut] = a[rng.integers(0, len(a), int(mut.sum()))]
    return x


def random_rows(N, L, seed):
    rng = np.random.default_rng(seed)
    a = np.frombuffer(b"AGCU-X", np.uint8)
    return a[rng.choice(6, (N, L), p=[.22, .22, .22, .22, .1, .02])]


def identical_rows(N, L, seed):
    return np.repeat(random_rows(1, L, seed), N, axis=0)


def copies_of_row0(N, L, seed):
    """About half the rows are row 0 again: in "min" mode every such copy is at distance 0, a tie."""
    x = family(N, L, 3, 0.1, seed)
    rng = np.random.default_rng(seed + 1)
    x[rng.random(N) < 0.5] = x[0]
    return x


def tail_rows(N, L, seed, far):
    """A family in which the LAST row must be the first pick: rows 1 .. N-2 sit at distance 2 .. L-1 from row 0 (all
    'A'), row N-1 at distance 1 (``far=False``: the unique nearest, "min" picks it) or L (``far=True``: the unique
    farthest, "max" picks it).  A kernel whose grid-stride or candidate loop stops before the last row picks another."""
    x = family(N, L, 4, 0.08, seed)
    x[0] = ord("A")
    x[1:N - 1, :2] = ord("G")
    x[1:N - 1, 2] = ord("A")
    x[N - 1] = ord("U") if far else ord("A")
    if not far:
        x[N - 1, 0] = ord("C")
    return x


class GreedyCase(NamedTuple):
    name: str            # the branch it targets
    kind: str            # builder
    N: int
    L: int
    num: int
    seed: int

    def chars(self):
        if self.kind == "family":
            return family(self.N, self.L, 4, 0.08, self.seed)
        if self.kind == "family_dense":
            return family(self.N, self.L, 4, 0.1, self.seed)
        if self.kind == "family_wide":
            return family(self.N, self.L, 6, 0.08, self.seed)
        if self.kind.startswith("tail"):
            return tail_rows(self.N, self.L, self.seed, far=self.kind == "tail_far")
        return {"random": random_rows, "identical": identical_rows, "copies": copies_of_row0}[self.kind](
            self.N, self.L, self.seed)


GREEDY_CASES = [
    # grid-stride of greedy_hamming_kernel (N > 592 * 8), more than one candidate per pick lane (N > 32 * 256) and
    # the grid-stride of greedy_mean_kernel (N > 592 * 256); past each edge the last row alone must be picked first
    GreedyCase("hamming_sweep_edge", "family", 4736, 24, 9, 1),
    GreedyCase("hamming_two_sweeps", "family", 4737, 24, 9, 2),
    GreedyCase("hamming_two_sweeps_near", "tail_near", 4737, 24, 9, 2),
    GreedyCase("hamming_two_sweeps_far", "tail_far", 4737, 24, 9, 2),
    GreedyCase("pick_two_per_lane_near", "tail_near", 8193, 24, 8, 3),
    GreedyCase("pick_two_per_lane_far", "tail_far", 8193, 24, 8, 3),
    GreedyCase("mean_two_sweeps_near", "tail_near", 151553, 12, 5, 4),
    GreedyCase("mean_two_sweeps_far", "tail_far", 151553, 12, 5, 4),
    # row length: one lane, a warp's stride edges, the dynamic shared LUT above 48 KiB, the longest accepted row
    GreedyCase("L1", "random", 300, 1, 9, 5),
    GreedyCase("L31", "family", 300, 31, 9, 6),
    GreedyCase("L32", "family", 300, 32, 9, 7),
    GreedyCase("L33", "family", 300, 33, 9, 8),
    GreedyCase("L6143", "random", 48, 6143, 9, 9),
    GreedyCase("L6144_big_lut", "random", 48, 6144, 9, 10),
    GreedyCase("L25599_max_lut", "random", 40, 25599, 9, 11),
    # ties everywhere
    GreedyCase("identical", "identical", 200, 20, 40, 12),
    GreedyCase("copies_of_row0", "copies", 400, 30, 150, 13),
    # pick counts: no round, the 8-accumulator edges, the recursion, a full sort block, all but one row
    GreedyCase("num1", "family", 300, 20, 1, 14),
    GreedyCase("num2", "family", 300, 20, 2, 15),
    GreedyCase("num8", "family", 300, 20, 8, 16),
    GreedyCase("num9", "family", 300, 20, 9, 17),
    GreedyCase("num128", "family", 600, 20, 128, 18),
    GreedyCase("num129", "family", 600, 20, 129, 19),
    GreedyCase("num136_recursion", "family", 600, 20, 136, 20),
    GreedyCase("num137_recursion", "family", 600, 20, 137, 21),
    GreedyCase("num1023", "family", 2000, 16, 1023, 22),
    GreedyCase("num1024_full_sort", "family", 2000, 16, 1024, 23),
    GreedyCase("num_all_but_one", "family", 300, 20, 299, 24),
    # deep selections whose outcome depends on the summation order (see SEPARATING)
    GreedyCase("separate_max", "family_dense", 600, 12, 200, 20),
    GreedyCase("separate_min", "family_wide", 1000, 20, 300, 20),
]

# the cases in which a sequential sum of the means selects another set of rows, and in which, from the oracle's own
# picks, a round at k > 128 would pick another row with it (checked on the CPU)
SEPARATING = {"max": "separate_max", "min": "separate_min"}


def kernel_sum_replay(counts, L, sequential=False):
    """Mean over axis 0 of ``counts / L`` (counts: mismatches [k, ...] against the k picks), float64, with the
    additions of ingest.cu's ``np_pairwise_sum`` in its order -- numpy's 8-accumulator pairwise sum: fewer than 8
    terms sequential from 0.0; up to 128 eight running sums over blocks of 8, tree-combined, then the tail; above 128
    split at n/2 rounded down to a multiple of 8 and recurse -- then divided by k.  Vectorised over the trailing axes;
    each element sees exactly the kernel's float64 operations.  ``sequential``: plain left-to-right sum instead."""
    v = np.asarray(counts, dtype=np.float64) / np.float64(L)           # lut[m] = (double)m / (double)L
    k = v.shape[0]
    if sequential:
        res = np.zeros(v.shape[1:])
        for i in range(k):
            res = res + v[i]
        return res / np.float64(k)
    return _pairwise(v) / np.float64(k)


def _pairwise(a):
    n = a.shape[0]
    if n < 8:
        res = np.zeros(a.shape[1:])
        for i in range(n):
            res = res + a[i]
        return res
    if n <= 128:
        r = [a[j].copy() for j in range(8)]
        i = 8
        while i < n - n % 8:
            for j in range(8):
                r[j] = r[j] + a[i + j]
            i += 8
        res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
        while i < n:
            res = res + a[i]
            i += 1
        return res
    n2 = n // 2
    n2 -= n2 % 8
    return _pairwise(a[:n2]) + _pairwise(a[n2:])


def greedy_trace(chars, num, mode, sequential=False, compare_from=None):
    """MSA.greedy_select's picks in the order they are made, with the means of kernel_sum_replay.  With
    ``compare_from=k0`` also returns the rounds k >= k0 at which, from the same picks, the other summation order
    (sequential for the kernel's, and vice versa) would pick another row: ``[(k, pick, other_pick)]``."""
    N, L = chars.shape
    picks = [0]
    taken = np.zeros(N, bool)
    taken[0] = True
    counts = np.empty((max(num - 1, 1), N), np.uint16)
    split = []
    bad = -np.inf if mode == "max" else np.inf
    opt = np.argmax if mode == "max" else np.argmin
    for k in range(1, num):
        counts[k - 1] = (chars != chars[picks[-1]]).sum(1)
        mean = kernel_sum_replay(counts[:k], L, sequential)
        mean[taken] = bad
        pick = int(opt(mean))
        if compare_from is not None and k >= compare_from:
            other = kernel_sum_replay(counts[:k], L, not sequential)
            other[taken] = bad
            if int(opt(other)) != pick:
                split.append((k, pick, int(opt(other))))
        picks.append(pick)
        taken[pick] = True
    return (picks, split) if compare_from is not None else picks


# ---------------------------------------------------------------------------------------------------- tokenize

def vocab_lut():
    """ingest_msa's 256-entry LUT: <unk> everywhere, the single-character tokens of the RNA alphabet at their bytes."""
    lut = np.full(256, I.RNA_TOKS.index("<unk>"), np.uint8)
    for i, t in enumerate(I.RNA_TOKS):
        if len(t) == 1:
            lut[ord(t)] = i
    return lut


def all_bytes_chars(R, L, seed):
    """uint8 [R, L] in which every byte value 0..255 occurs (row 0 starts with 0, 1, ..., 255 when L allows)."""
    rng = np.random.default_rng(seed)
    x = rng.integers(0, 256, (R, L), dtype=np.uint8)
    flat = x.reshape(-1)
    flat[:min(256, flat.size)] = np.arange(min(256, flat.size), dtype=np.uint8)
    return x


def tokenize_reference(chars, rows, lut, bos):
    sel = chars if rows is None else chars[np.asarray(rows)]
    out = np.empty((sel.shape[0], sel.shape[1] + 1), np.int64)
    out[:, 0] = bos
    out[:, 1:] = lut[sel]
    return out


# (R, L, with rows): R not a multiple of 8, L across 32-lane strides
TOKENIZE_CASES = [(1, 1, False), (7, 31, True), (8, 32, False), (9, 33, True), (13, 256, False), (13, 256, True),
                  (100, 65, True), (1000, 300, False), (4097, 40, True)]


# ---------------------------------------------------------------------------------------------------- packs

SS_CODES = {"A": 0, "C": 1, "G": 2, "U": 3}          # inference._SEQ_CODES: anything else is 255 (an all-zero one-hot)


def seq_codes(seq):
    return np.array([SS_CODES.get(ch, 255) for ch in seq], np.uint8)


def pack_sequence(L, seed):
    """Mostly ACGU, with X, N, '-', lowercase and T (all outside the one-hot) mixed in."""
    rng = np.random.default_rng(seed)
    return "".join(rng.choice(list("ACGUACGUACGUXN-acgT"), L))


def ss_reference(atp, seq):
    """[1, 8 + K, L, L] float32: the outer concatenation of the ACGU one-hot (channels 0-3: seq[i], 4-7: seq[j]) in
    front of the maps, as oracle/gen_golden_ss.py runs the SS pre-processing (outer_concatenation, feature_load's
    concatenate, format_input_shape's transpose).  Non-ACGU letters have an all-zero one-hot."""
    L = len(seq)
    oh = np.array([[1.0 if ch == a else 0.0 for a in "ACGU"] for ch in seq], np.float32).reshape(L, 4)
    pair = np.concatenate([np.broadcast_to(oh[:, None, :], (L, L, 4)), np.broadcast_to(oh[None, :, :], (L, L, 4))], 2)
    x = np.concatenate([pair, np.asarray(atp, np.float32).transpose(1, 2, 0)], axis=2)
    return np.ascontiguousarray(np.transpose(x[None], (0, 3, 1, 2)))


# (L, start, K): one block column, 255/256/257 around the 256-thread block (grid.x > 1), two extra blocks
SS_CASES = [(L, s, K) for L in (1, 255, 256, 257, 513) for s in (0, 1) for K in (1, 120) if not (L == 513 and K == 120 and s)]


def rsa_reference(emb, D, seq, mu, sd, mu_oh=None, sd_oh=None):
    """oracle.msa_ref.rsa_input on the first D features of ``emb`` [L, ld]: [1, n_oh + D + 1, L] float32."""
    return O.rsa_input(np.ascontiguousarray(emb[:, :D]), seq, mu, sd, mu_oh, sd_oh)


RSA_CASES = [(L, D, oh, extra) for D in (1, 27, 31, 32, 33, 768) for oh in (False, True) for extra in (0, 5)
             for L in (1, 31, 32, 33, 257)]


def rsa_inputs(L, D, extra, seed):
    """emb [L, D + extra] (the extra columns NaN: they must never be read), positive stds, and one-hot statistics."""
    rng = np.random.default_rng(seed)
    emb = np.full((L, D + extra), np.nan, np.float32)
    emb[:, :D] = (rng.standard_normal((L, D)) * 0.7).astype(np.float32)
    mu = (rng.standard_normal(D) * 0.1).astype(np.float32)
    sd = rng.uniform(0.2, 1.5, D).astype(np.float32)
    mu_oh = rng.uniform(0.15, 0.35, 4)
    sd_oh = rng.uniform(0.35, 0.5, 4)
    return emb, mu, sd, mu_oh, sd_oh
