"""CPU checks of tests/ingest_cases.py: the restatements reproduce every golden of the ingest and the packs, the SeqIO
restatement reads hand-written files as spelled out here, every alignment builder reaches the launch branch it is
named for, the kernel's summation order equals numpy's mean bit for bit, and the deep cases really separate it from a
sequential sum.  (The GPU side is tests/test_gpu_ingest_edges.py.)"""
import os

import numpy as np
import pytest

import ingest_cases as IC
from oracle import msa_ingest_ref as I
from rnamsm_b200.ingest import cleaned_length, split_records

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = {c.name: c for c in IC.GREEDY_CASES}


# ------------------------------------------------------------------------------------------------ goldens

@pytest.mark.parametrize("name", ["rand", "dups", "deep", "2drb"])
@pytest.mark.parametrize("mode", ["max", "min"])
def test_trace_reproduces_ingest_golden(name, mode):
    g = np.load(os.path.join(GOLDEN, "ingest.npz"))
    if name == "2drb" and mode == "min":
        pytest.skip("the golden has no min-mode vector for 2DRB_1")
    num = 512 if name == "2drb" else int(g[f"{name}_num"])
    assert sorted(IC.greedy_trace(g[f"{name}_chars"], num, mode)) == g[f"{name}_{mode}_idx"].tolist()


def test_ss_restatement_reproduces_golden():
    g = np.load(os.path.join(GOLDEN, "ss_pack.npz"))
    x = IC.ss_reference(g["atp"], str(g["seq"]))
    assert x.dtype == g["x"].dtype and np.array_equal(x, g["x"])


def test_rsa_reference_reproduces_golden():
    g = np.load(os.path.join(GOLDEN, "rsa_pack.npz"))
    emb = np.concatenate([g["emb"], np.full((g["emb"].shape[0], 5), np.nan, np.float32)], 1)
    x = IC.rsa_reference(emb, 768, str(g["seq"]), g["mu_emb"], g["std_emb"], g["mu_oh"], g["std_oh"])
    assert x.dtype == g["x"].dtype and np.array_equal(x, g["x"])


# ------------------------------------------------------------------------------------------------ FASTA restatement

def test_seqio_restatement_on_hand_written_files():
    """Universal newlines, per-line rstrip(), then ' ' and '\\r' removed from the joined sequence."""
    f = (b"junk before\r\n>x >y\r\nAC\tG U\x0b\r\nac.\x0c\t\x1f \n"    # tab inside a line kept; trailing \v \f \t dropped
         b">e\n"                                                          # empty record
         b">b\rAC\rGU \t\r>c\x0c\nA\x0cC\n \n\t\n"                        # lone '\r' line ends, '\r>' starts a record
         b">last\nAC\x1cGU")                                              # no newline at the end of the file
    assert IC.seqio_records(f) == [("x >y", "AC\tGUac."), ("e", ""), ("b", "ACGU"), ("c", "A\x0cC"), ("last", "AC\x1cGU")]
    assert IC.reference_rows(f) == ["AC\tGU", "", "ACGU", "A\x0cC", "AC\x1cGU"]
    assert IC.seqio_records(b"no record here\n") == []
    assert IC.seqio_records(b">only\n") == [("only", "")]
    assert IC.reference_rows(b">t\nAtTgu.*NRY-\n") == ["AUXXX-"]


@pytest.mark.parametrize("name", sorted(IC.messy_files()))
def test_split_records_and_cleaned_length_follow_seqio(name, tmp_path):
    """split_records finds SeqIO's records and cleaned_length gives every record's length; a well-formed file
    cleans every record to the first record's length."""
    data, well_formed = IC.messy_files()[name]
    p = tmp_path / "x.a2m"
    p.write_bytes(data)
    headers, raw, off = split_records(str(p))
    recs = IC.seqio_records(data)
    rows = IC.reference_rows(data)
    assert headers == [t.strip() for t, _ in recs]
    assert [cleaned_length(raw[off[i]:off[i + 1]]) for i in range(len(rows))] == [len(r) for r in rows]
    assert (len({len(r) for r in rows}) == 1) == well_formed
    if name == "malformed":
        assert {len(r) for r in rows} >= {0, 20, 25, 19}


def test_writer_round_trips_rows():
    """write_messy's noise is exactly what SeqIO + from_fasta drop: the rows come back (tabs inside lines included)."""
    rng = np.random.default_rng(1)
    rows = ["AGX\tU-\x0bCX\x1cA", "UUUU\x0c\tGGGGAA", "A" * 13]
    for ends in ("lf", "crlf", "cr", "mixed"):
        data = IC.write_messy(rows, rng, ends=ends, width=3, trailing=" \t\x0b\x0c\x1f")
        assert IC.reference_rows(data) == rows


def test_chunk_edge_file_reaches_every_body_length(tmp_path):
    data = IC.chunk_edge_file()
    rows = IC.reference_rows(data)
    assert {len(r) for r in rows} == {16}
    assert sum("\t" in r for r in rows) == 10                    # the runs followed by text keep their tabs
    p = tmp_path / "x.a2m"
    p.write_bytes(data)
    _, _, off = split_records(str(p))
    assert {31, 32, 33, 63, 64, 65, 1023, 1024, 1025} <= set(np.diff(off).tolist())


# ------------------------------------------------------------------------------------------------ greedy select

def test_builders_reach_their_branches():
    g = {c.name: IC.launch_geometry(c.N, c.L, c.num) for c in IC.GREEDY_CASES}
    assert g["hamming_sweep_edge"]["hamming_sweeps"] == 1 and g["hamming_two_sweeps"]["hamming_sweeps"] == 2
    assert g["pick_two_per_lane_far"]["pick_per_lane"] == 2 and g["hamming_two_sweeps"]["pick_per_lane"] == 1
    assert g["mean_two_sweeps_far"]["mean_sweeps"] == 2 and g["pick_two_per_lane_far"]["mean_sweeps"] == 1
    assert not g["L6143"]["big_lut"] and g["L6144_big_lut"]["big_lut"]
    assert g["L25599_max_lut"]["lut_bytes"] == 200 * 1024
    assert g["num128"]["max_k"] == 127 and g["num129"]["max_k"] == 128 and not g["num129"]["recursion"]
    assert g["num136_recursion"]["recursion"] and g["num137_recursion"]["max_k"] == 136
    assert g["num1024_full_sort"]["sort_threads_used"] == 1024 and g["num1"]["max_k"] == 0
    assert CASES["num_all_but_one"].num == CASES["num_all_but_one"].N - 1
    for c in IC.GREEDY_CASES:
        x = c.chars()
        assert x.shape == (c.N, c.L) and x.dtype == np.uint8 and 1 <= c.num <= min(c.N, 1024)
        assert c.num <= 137 or c.N <= 2000, "the CPU oracle costs num^2 * N"


@pytest.mark.parametrize("name", [c.name for c in IC.GREEDY_CASES if c.kind.startswith("tail")])
def test_tail_cases_pick_the_row_past_the_edge_first(name):
    """The last row lies past the first hamming sweep (row 4736), in pick lane 0's second candidate block (block 32)
    or past the first mean sweep (row 151552), and the oracle picks it in round 1."""
    c = CASES[name]
    mode = "max" if c.kind == "tail_far" else "min"
    x = c.chars()
    assert IC.greedy_trace(x, 2, mode) == [0, c.N - 1]
    assert c.N - 1 in I.greedy_select_indices(x, c.num, mode)
    g = IC.launch_geometry(c.N, c.L, c.num)
    assert g["hamming_sweeps"] == 2 or g["pick_per_lane"] == 2 or g["mean_sweeps"] == 2


def test_tie_builders_tie():
    x = CASES["identical"].chars()
    assert (x == x[0]).all()
    x = CASES["copies_of_row0"].chars()
    assert (x == x[0]).all(1).sum() > CASES["copies_of_row0"].num        # distance-0 ties through every min round
    x = CASES["num137_recursion"].chars()
    assert len(np.unique(x, axis=0)) < x.shape[0]                         # duplicate rows in the family


def test_kernel_sum_replay_is_numpy_mean_for_every_k():
    """The reference's np.delete(pairwise_distances, indices, axis=1).mean(0) for k = 1 .. 1023 picks (k rows, k
    deleted columns), bit for bit; the sequential variant differs for most k."""
    rng = np.random.default_rng(0)
    L, N = 37, 1100
    seq_differs = 0
    for k in range(1, 1024):
        counts = rng.integers(0, L + 1, (k, N)).astype(np.uint16)
        pd = counts / np.float64(L)
        idx = rng.choice(N, k, replace=False)
        want = np.delete(pd, idx, axis=1).mean(0)
        got = np.delete(IC.kernel_sum_replay(counts, L), idx)
        assert np.array_equal(got, want), k
        seq_differs += not np.array_equal(np.delete(IC.kernel_sum_replay(counts, L, sequential=True), idx), want)
    assert seq_differs > 900


def test_hamming_counts_are_cdist():
    """kernel_sum_replay's lut[m] = m / L is scipy's cdist(..., "hamming") value exactly."""
    from scipy.spatial.distance import cdist
    for c in (CASES["L33"], CASES["num137_recursion"]):
        x = c.chars()
        d = cdist(x[3:4], x, "hamming")[0]
        assert np.array_equal(d, (x != x[3]).sum(1).astype(np.float64) / np.float64(c.L))


@pytest.mark.parametrize("name", [c.name for c in IC.GREEDY_CASES if c.N <= 2000 and c.num <= 300])
@pytest.mark.parametrize("mode", ["max", "min"])
def test_trace_equals_oracle(name, mode):
    c = CASES[name]
    x = c.chars()
    assert sorted(IC.greedy_trace(x, c.num, mode)) == I.greedy_select_indices(x, c.num, mode)


@pytest.mark.parametrize("mode", ["max", "min"])
def test_deep_cases_separate_the_summation_orders(mode):
    """A sequential sum of the means ends with another set of rows, and from the oracle's own picks a round at
    k > 128 (the recursion) picks another row with it: a kernel that lost the pairwise order fails the GPU test
    instead of agreeing by luck."""
    c = CASES[IC.SEPARATING[mode]]
    x = c.chars()
    want = I.greedy_select_indices(x, c.num, mode)
    picks, split = IC.greedy_trace(x, c.num, mode, compare_from=129)
    assert sorted(picks) == want
    assert split, f"{c.name} {mode}: no round at k > 128 separates the orders"
    k, pick, other = split[0]
    print(f"{c.name} {mode}: round k={k} picks row {pick} (pairwise), a sequential sum would pick row {other}; "
          f"{len(split)} such rounds")
    assert pick != other and k > 128
    seq = sorted(IC.greedy_trace(x, c.num, mode, sequential=True))
    assert seq != want
    print(f"{c.name} {mode}: sequential sums select {len(set(seq) - set(want))} other rows")


# ------------------------------------------------------------------------------------------------ tokenize / packs

def test_tokenize_reference_is_encode():
    lut = IC.vocab_lut()
    x = IC.all_bytes_chars(3, 300, 1)
    assert set(np.unique(x).tolist()) == set(range(256))
    want = I.encode([bytes(r).decode("latin-1") for r in x])
    assert np.array_equal(IC.tokenize_reference(x, None, lut, 0), want)
    assert np.array_equal(IC.tokenize_reference(x, [2, 0], lut, 0), want[[2, 0]])


def test_pack_cases_cover_the_edges():
    assert {L for L, _, _ in IC.SS_CASES} == {1, 255, 256, 257, 513}
    assert {(s, K) for _, s, K in IC.SS_CASES} == {(0, 1), (0, 120), (1, 1), (1, 120)}
    chans = {(oh * 4 + D + 1) % 32 for _, D, oh, _ in IC.RSA_CASES}
    assert {0, 1} <= chans                                                # n_oh + D + 1 across multiples of 32
    assert any(not oh and D % 2 for _, D, oh, _ in IC.RSA_CASES)
    seq = IC.pack_sequence(400, 1)
    assert set("XN-acgT") <= set(seq) and (IC.seq_codes(seq) == 255).any()
    emb, *_ = IC.rsa_inputs(3, 4, 5, 0)
    assert np.isnan(emb[:, 4:]).all() and not np.isnan(emb[:, :4]).any()
