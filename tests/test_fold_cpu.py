"""CPU: the float32 restatement of the folding (tests/fold_ref.py) against brute force and hand-built structures, the
structure files, and the argument handling of ``fold_pairs`` and ``python -m rnamsm_b200.fold``."""
import numpy as np
import pytest

import fold_ref as F


def random_map(L, seed, quant=None):
    rng = np.random.default_rng(seed)
    S = rng.random((L, L)).astype(np.float32) / np.float32(max(L, 1) / 4)
    if quant:
        S = (np.round(S * quant) / quant).astype(np.float32)
    return S


def random_seq(L, seed):
    rng = np.random.default_rng(seed)
    return "".join(rng.choice(list("AGCUAGCUXN-"), size=L))


def planted(L, helices, noise=None, seed=0, value=0.9):
    """Map with stems (i, j, n): pairs (i + t, j - t), t < n, at `value` over uniform noise below `noise` (default
    0.2 / L, so every row of probabilities sums below 1)."""
    rng = np.random.default_rng(seed)
    noise = 0.2 / L if noise is None else noise
    S = (rng.random((L, L)) * noise).astype(np.float32)
    want = np.full(L, -1, dtype=np.int32)
    for i, j, n in helices:
        for t in range(n):
            S[i + t, j - t] = value
            want[i + t], want[j - t] = j - t, i + t
    return S, want


@pytest.mark.parametrize("L", range(1, 13))
@pytest.mark.parametrize("mode", ["mea", "score"])
def test_restatement_equals_brute_force(L, mode):
    for seed in range(3):
        S = random_map(L, 100 * L + seed)
        if mode == "score":
            S = (S - np.float32(0.5 / max(L, 1) * 4)).astype(np.float32)       # negative scores too
        kw = dict(mode=mode, gamma=1.5, threshold=-1.0 if mode == "score" else 0.0, min_loop=seed % 2 * 3)
        w, u = F.weights(S, **kw)
        pairs, score = F.fold(S, **kw)
        best = F.brute_force(w, u)
        assert abs(float(score) - best) <= 1e-6 * max(1.0, abs(best)), (L, seed, score, best)
        assert abs(F.structure_score(w, u, pairs) - float(score)) <= 1e-6 * max(1.0, abs(best))
        for i, k in enumerate(pairs):
            assert k == -1 or (pairs[k] == i and np.isfinite(w[min(i, k), max(i, k)]))


def test_brute_force_counts_nested_structures():
    ok = np.triu(np.ones((6, 6), dtype=bool), 1)
    assert len(F.nested_structures(ok)) == 51                        # Motzkin number M_6
    ok = np.triu(np.ones((6, 6), dtype=bool), 4)                      # j - i > 3
    assert len(F.nested_structures(ok)) == 1 + 3 + 0


@pytest.mark.parametrize("mode", ["mea", "score"])
def test_hairpin_folds_as_drawn(mode):
    S, want = planted(30, [(2, 27, 8)])
    pairs, _ = F.fold(S, mode=mode, threshold=0.5 if mode == "score" else 0.0)
    assert np.array_equal(pairs, want)


def test_two_helix_junction_folds_as_drawn():
    S, want = planted(60, [(0, 59, 5), (6, 25, 6), (28, 52, 7)])
    pairs, _ = F.fold(S, mode="mea")
    assert np.array_equal(pairs, want)
    pairs, _ = F.fold(S, mode="score", threshold=0.5)
    assert np.array_equal(pairs, want)


def test_canonical_and_min_loop_rules():
    S = np.zeros((12, 12), dtype=np.float32)
    S[0, 11] = S[1, 10] = S[2, 9] = S[3, 4] = 0.9
    seq = "GCAAAAAAAAUC"                 # G-C pairs, C-U does not, A-A does not
    pairs, _ = F.fold(S, seq, mode="mea", min_loop=0)
    assert pairs[0] == 11 and pairs[1] == -1 and pairs[2] == -1 and pairs[3] == -1
    pairs, _ = F.fold(S, seq, mode="mea", min_loop=0, canonical=False)
    assert pairs[0] == 11 and pairs[1] == 10 and pairs[2] == 9 and pairs[3] == 4
    pairs, _ = F.fold(S, seq, mode="mea", min_loop=3, canonical=False)
    assert pairs[3] == -1 and pairs[0] == 11
    for letters in ("XG", "NC", "-G", "AA", "CC"):
        assert not F.allowed(np.ones((6, 6), np.float32), letters[0] + "AAAA" + letters[1], min_loop=0)[0, 5]
    for letters in ("AU", "UA", "GC", "CG", "GU", "UG"):
        assert F.allowed(np.ones((6, 6), np.float32), letters[0] + "AAAA" + letters[1], min_loop=0)[0, 5]


def test_ties_break_to_unpaired_then_nearest_partner():
    S = np.full((8, 8), 0.25, dtype=np.float32)
    pairs, score = F.fold(S, mode="score", min_loop=0, threshold=0.0)
    # every pair scores 0.25; 4 pairs at most; i = 0 cannot be left unpaired without losing a pair
    assert pairs.tolist() == [1, 0, 3, 2, 5, 4, 7, 6] and score == np.float32(1.0)
    pairs, score = F.fold(np.zeros((5, 5), np.float32), mode="score", threshold=-1.0, min_loop=0)
    assert (pairs == -1).all() and score == 0.0                      # 0-weight pairs tie with unpaired


def test_nonfinite_map_is_an_error():
    S = random_map(10, 1)
    S[2, 7] = np.nan
    with pytest.raises(ValueError):
        F.fold(S)
    S = random_map(10, 1)
    S[7, 2] = np.inf                                                   # lower triangle: not read
    F.fold(S, mode="score")


def parse_dot_bracket(db):
    stack, pairs = [], [-1] * len(db)
    for i, ch in enumerate(db):
        if ch == "(":
            stack.append(i)
        elif ch == ")":
            k = stack.pop()
            pairs[i], pairs[k] = k, i
    assert not stack
    return pairs


def parse_ct(path):
    lines = open(path).read().splitlines()
    n, name = lines[0].split("\t", 1)
    seq, pairs = "", []
    for t, line in enumerate(lines[1:]):
        f = line.split("\t")
        assert int(f[0]) == t + 1 and int(f[2]) == t and int(f[3]) == (t + 2 if t + 1 < int(n) else 0)
        assert int(f[5]) == t + 1
        seq += f[1]
        pairs.append(int(f[4]) - 1)
    assert len(pairs) == int(n)
    return name, seq, pairs


def parse_bpseq(path):
    seq, pairs = "", []
    for t, line in enumerate(open(path).read().splitlines()):
        i, b, k = line.split()
        assert int(i) == t + 1
        seq += b
        pairs.append(int(k) - 1)
    return seq, pairs


def test_structure_files_round_trip(tmp_path):
    from rnamsm_b200 import structure as ST
    S, want = planted(40, [(1, 38, 6), (9, 30, 4)])
    pairs, _ = F.fold(S)
    seq = random_seq(40, 3)
    db = ST.dot_bracket(pairs)
    assert db.count("(") == 10 and parse_dot_bracket(db) == pairs.tolist()
    ST.write_ct(str(tmp_path / "x.ct"), "query 1", seq, pairs)
    assert parse_ct(tmp_path / "x.ct") == ("query 1", seq, pairs.tolist())
    ST.write_bpseq(str(tmp_path / "x.bpseq"), seq, pairs)
    assert parse_bpseq(tmp_path / "x.bpseq") == (seq, pairs.tolist())
    assert ST.dot_bracket(np.full(3, -1)) == "..."
    for bad in ([1, -1, -1], [2, 2, 0], [5, -1]):
        with pytest.raises(ValueError):
            ST.dot_bracket(bad)
    with pytest.raises(ValueError):
        ST.write_bpseq(str(tmp_path / "y"), "AC", pairs)


def test_fold_pairs_argument_errors_before_the_device():
    import torch
    from rnamsm_b200 import structure as ST
    S = torch.zeros((6, 6))
    for kw, match in ((dict(mode="x"), "mode"), (dict(gamma=0.0), "gamma"), (dict(gamma=float("nan")), "gamma"),
                      (dict(gamma=1e39), "gamma"), (dict(threshold=float("inf")), "threshold"),
                      (dict(threshold=1e39), "threshold"), (dict(min_loop=-1), "min_loop"),
                      (dict(min_loop=1.5), "min_loop"), (dict(canonical=True), "sequences"),
                      (dict(sequences="AGCUA"), "letters"), (dict(sequences="AGCUAT"), "outside"),
                      (dict(sequences=["AGCUAA", "AGCUAA"]), "one sequence")):
        with pytest.raises(ValueError, match=match):
            ST.fold_pairs(S, **kw)
    for bad in (torch.zeros(6), torch.zeros((6, 5)), torch.zeros((6, 6), dtype=torch.float64), torch.zeros((0, 0))):
        with pytest.raises(ValueError):
            ST.fold_pairs(bad)
    with pytest.raises(ValueError):
        ST.fold_pairs([])
    with pytest.raises(RuntimeError, match="CUDA"):                  # gamma is not read in score mode
        ST.fold_pairs(S, mode="score", gamma=0.0)
    with pytest.raises(RuntimeError, match="CUDA"):
        ST.fold_pairs([S, torch.zeros((3, 3))], ["AGCUAG", "GGC"])


def test_workspace_bytes_is_host_math():
    import ctypes as C
    from rnamsm_b200 import _lib as L

    def size(*Ls):
        return L.lib.rnamsm_fold_workspace_bytes(len(Ls), (C.c_int * len(Ls))(*Ls))

    assert size(0) == 0 and b"L = 0" in L.lib.rnamsm_last_error()
    assert L.lib.rnamsm_fold_workspace_bytes(0, None) == 0
    one = size(100)                                                    # T = 32: Lp = 128, ld = 132
    assert one % 256 == 0 and 2 * 128 * 132 * 4 < one < 2 * 128 * 132 * 4 + 16384   # + split-K partials
    assert size(100, 50) > one
    big = size(200_000)
    assert big > 2 * 200_000 ** 2 * 4                                  # about 320 GB of tables


def test_cli_parses_arguments():
    from rnamsm_b200 import fold
    a = fold.parse_args(["--MSA_file", "x", "--out_prefix", "p", "--source", "dca"])
    assert a.mode == "score" and a.gamma == 1.0 and a.min_loop == 3 and not a.no_canonical
    a = fold.parse_args(["--MSA_file", "x", "--out_prefix", "p", "--source", "contact-head"])
    assert a.mode == "mea" and a.precision == "fp16"
    a = fold.parse_args(["--MSA_file", "x", "--out_prefix", "p", "--source", "npy", "--map", "m.npy", "--mode",
                         "score", "--threshold", "0.2", "--min_loop", "0", "--no_canonical", "--gamma", "4"])
    assert (a.mode, a.threshold, a.min_loop, a.no_canonical, a.gamma, a.map) == ("score", 0.2, 0, True, 4.0, "m.npy")
    assert fold.parse_args(["--MSA_file", "x", "--out_prefix", "p", "--source", "jacobian"]).mode == "score"


@pytest.mark.parametrize("argv", [
    ["--out_prefix", "p", "--source", "dca"],
    ["--MSA_file", "x", "--source", "dca"],
    ["--MSA_file", "x", "--out_prefix", "p"],
    ["--MSA_file", "x", "--out_prefix", "p", "--source", "rosetta"],
    ["--MSA_file", "x", "--out_prefix", "p", "--source", "npy"],
    ["--MSA_file", "x", "--out_prefix", "p", "--source", "dca", "--map", "m.npy"],
    ["--MSA_file", "x", "--out_prefix", "p", "--source", "dca", "--gamma", "0"],
    ["--MSA_file", "x", "--out_prefix", "p", "--source", "dca", "--min_loop", "-1"],
    ["--MSA_file", "x", "--out_prefix", "p", "--source", "dca", "--threshold", "nan"],
    ["--MSA_file", "x", "--out_prefix", "p", "--source", "dca", "--mode", "mfe"],
])
def test_cli_argument_errors(argv):
    from rnamsm_b200 import fold
    with pytest.raises(SystemExit):
        fold.parse_args(argv)
