"""GPU: nested secondary structure from a pair map (``rnamsm_b200.fold_pairs``, ``rnamsm_fold``,
``python -m rnamsm_b200.fold``) against the float32 restatement of tests/fold_ref.py.

Every table entry is one fp32 add and max is exact, so scores are equal as fp32 values and pairs identical, at every
length, both tile sizes, both modes, on tie-heavy maps, in ragged batches and across repeated calls."""
import sys

import numpy as np
import pytest
import torch

import fold_ref as F

pytestmark = pytest.mark.gpu

LENGTHS = [1, 2, 4, 5, 31, 32, 33, 63, 64, 65, 127, 128, 129, 200, 513, 1000, 2048]


@pytest.fixture(scope="module")
def pkg():
    import rnamsm_b200
    return rnamsm_b200


def prob_map(L, seed, quant=None):
    """Symmetric map of pair probabilities whose rows sum to at most 0.8; with quant, a sparse map of multiples of
    1 / quant in [0, 1] instead."""
    rng = np.random.default_rng(seed)
    if quant:
        S = rng.integers(0, quant + 1, size=(L, L)) / quant * (rng.random((L, L)) < 4.0 / L)
        return S.astype(np.float32)
    S = rng.random((L, L)) ** 4
    S = S + S.T
    S = S / max(1e-30, S.sum(axis=1).max()) * 0.8
    return S.astype(np.float32)


def score_map(L, seed, quant=None):
    rng = np.random.default_rng(seed)
    S = rng.standard_normal((L, L))
    if quant:
        S = np.round(S * quant) / quant
    return S.astype(np.float32)


def random_seq(L, seed):
    rng = np.random.default_rng(seed)
    return "".join(rng.choice(list("AGCUAGCUAGCUXN-"), size=L))


def launches():
    torch.cuda.synchronize()
    from rnamsm_b200 import _lib
    return _lib.lib.rnamsm_launch_count()


def check(pkg, S, seq=None, **kw):
    pairs, score = pkg.fold_pairs(torch.from_numpy(S).cuda(), seq, **kw)
    ref_pairs, ref_score = F.fold(S, seq, **kw)
    assert pairs.dtype == torch.int32 and pairs.shape == (S.shape[0],) and pairs.is_cuda
    assert np.float32(score) == ref_score and isinstance(score, float)
    assert np.array_equal(pairs.cpu().numpy(), ref_pairs)
    return pairs, score


@pytest.mark.parametrize("L", LENGTHS)
def test_mea_matches_restatement(pkg, L):
    check(pkg, prob_map(L, L))


@pytest.mark.parametrize("L", LENGTHS)
def test_score_matches_restatement(pkg, L):
    check(pkg, score_map(L, L + 1), mode="score")


@pytest.mark.parametrize("L", [33, 129, 513])
@pytest.mark.parametrize("canonical", [False, True])
@pytest.mark.parametrize("min_loop", [0, 3])
@pytest.mark.parametrize("mode,gamma", [("mea", 0.5), ("mea", 1.0), ("mea", 4.0), ("score", 1.0)])
def test_parameter_grid(pkg, L, canonical, min_loop, mode, gamma):
    S = prob_map(L, 7 * L) if mode == "mea" else score_map(L, 7 * L)
    seq = random_seq(L, L)
    thr = 0.0 if mode == "mea" else -0.5
    check(pkg, S, seq, mode=mode, gamma=gamma, threshold=thr, min_loop=min_loop, canonical=canonical)


@pytest.mark.parametrize("L", [5, 33, 64, 129, 1000, 1100])
@pytest.mark.parametrize("mode", ["mea", "score"])
def test_tie_heavy_maps(pkg, L, mode):
    """Values on multiples of 1/8: many candidates tie exactly, so the tie rule decides the structure."""
    S = prob_map(L, 3 * L, quant=8) if mode == "mea" else score_map(L, 3 * L, quant=8)
    assert np.all(S * 8 == np.round(S * 8))
    check(pkg, S, mode=mode, min_loop=1)
    check(pkg, S, random_seq(L, 5), mode=mode, min_loop=0, threshold=-2.0)


def planted_device(L, seed):
    """fp32 [L, L] on the device: noise below 0.2 / L and nested stems at 0.9; and the planted pairs."""
    rng = np.random.default_rng(seed)
    want = np.full(L, -1, dtype=np.int64)
    g = torch.Generator(device="cuda").manual_seed(seed)
    S = torch.rand((L, L), device="cuda", generator=g) * (0.2 / L)
    i = 0
    while i < L - 40:                                # consecutive hairpins and two-stem junctions
        n = int(rng.integers(4, 12))
        span = int(rng.integers(2 * n + 6, min(2 * n + 300, L - i)))
        j = i + span - 1
        for t in range(n):
            want[i + t], want[j - t] = j - t, i + t
        inner = i + n + 2
        if j - n - 2 - inner > 2 * 5 + 8 and rng.random() < 0.5:
            m = 5
            for t in range(m):
                want[inner + t], want[j - n - 2 - t] = j - n - 2 - t, inner + t
        i = j + 1 + int(rng.integers(0, 5))
    idx = np.flatnonzero(want > np.arange(L))
    S[torch.from_numpy(idx).cuda(), torch.from_numpy(want[idx]).cuda()] = 0.9
    return S, want


@pytest.mark.parametrize("L", [4096, 8192])
def test_planted_helices_long(pkg, L):
    S, want = planted_device(L, L)
    pairs, score = pkg.fold_pairs(S, mode="mea", gamma=1.0)
    got = pairs.cpu().numpy()
    assert np.array_equal(got, want)
    S64 = S.double().cpu().numpy()
    up = np.triu(S64, 1)
    u = 1.0 - (up.sum(axis=1) + up.sum(axis=0))
    w = float(np.float32(2.0)) * S.cpu().numpy().astype(np.float64)
    ref = sum(w[i, k] for i, k in enumerate(got) if k > i) + u[got < 0].sum()
    print(f"L {L}: {int((got >= 0).sum()) // 2} pairs, score {score:.6f}, float64 {ref:.6f}")
    assert abs(score - ref) <= 1e-5 * abs(ref)
    again, score2 = pkg.fold_pairs(S, mode="mea", gamma=1.0)
    assert torch.equal(again, pairs) and score2 == score


def test_ragged_batch_bit_identical_to_single_maps(pkg):
    for Ls in ([300, 1, 65, 1000, 33, 32], [1100, 70, 2, 64, 129]):
        maps = [torch.from_numpy(prob_map(L, L + 11)).cuda() for L in Ls]
        seqs = [random_seq(L, L) for L in Ls]
        for kw in (dict(), dict(sequences=seqs, min_loop=0)):
            n0 = launches()
            pairs, scores = pkg.fold_pairs(maps, **kw)
            T = 32 if max(Ls) <= 1024 else 64
            assert launches() - n0 == 2 + -(-max(Ls) // T)
            assert len(pairs) == len(Ls) and len(scores) == len(Ls)
            for m, S in enumerate(maps):
                alone_kw = dict(kw)
                if "sequences" in kw:
                    alone_kw["sequences"] = seqs[m]
                p1, s1 = pkg.fold_pairs(S, **alone_kw)
                assert torch.equal(p1, pairs[m]) and s1 == scores[m]


@pytest.mark.parametrize("L", [1, 32, 33, 1024, 1025, 2048, 2049])
def test_launch_count_follows_formula(pkg, L):
    """prep + one fill launch per tile diagonal + traceback: 2 + ceil(L / T), T = 32 up to 1024, else 64."""
    S = torch.from_numpy(score_map(L, 1)).cuda()
    n0 = launches()
    pkg.fold_pairs(S, mode="score")
    T = 32 if L <= 1024 else 64
    assert launches() - n0 == 2 + -(-L // T)


def test_repeated_calls_same_bits(pkg):
    S = torch.from_numpy(prob_map(700, 9)).cuda()
    p0, s0 = pkg.fold_pairs(S)
    for _ in range(3):
        p, s = pkg.fold_pairs(S)
        assert torch.equal(p, p0) and s == s0


def test_nonfinite_map_raises(pkg):
    for bad in (float("nan"), float("inf"), -float("inf")):
        S = torch.from_numpy(prob_map(100, 2)).cuda()
        S[10, 70] = bad
        with pytest.raises(ValueError, match="non-finite"):
            pkg.fold_pairs(S)
        with pytest.raises(ValueError, match="non-finite"):
            pkg.fold_pairs([torch.from_numpy(prob_map(40, 1)).cuda(), S], mode="score")
    S = torch.from_numpy(prob_map(100, 2)).cuda()
    S[70, 10] = float("nan")                                            # lower triangle: not read
    check(pkg, S.cpu().numpy())
    S = torch.full((40, 40), 3e38, device="cuda")
    with pytest.raises(ValueError, match="overflows"):
        pkg.fold_pairs(S, gamma=1.0)


def test_bad_arguments_raise_with_no_launch(pkg):
    S = torch.from_numpy(prob_map(20, 2)).cuda()
    n0 = launches()
    for kw in (dict(mode="mfe"), dict(gamma=0.0), dict(gamma=-1.0), dict(threshold=float("nan")), dict(min_loop=-1),
               dict(canonical=True), dict(sequences="AGCU"), dict(sequences="B" * 20)):
        with pytest.raises(ValueError):
            pkg.fold_pairs(S, **kw)
    for bad in (S[:, :5], S.double(), S[0], [S, S.cpu()]):
        with pytest.raises((ValueError, RuntimeError)):
            pkg.fold_pairs(bad)
    with pytest.raises(RuntimeError, match="CUDA"):
        pkg.fold_pairs(S.cpu())
    assert launches() == n0
    from rnamsm_b200 import _lib as L
    import ctypes as C
    Ls = (C.c_int * 1)(20)
    nbytes = L.lib.rnamsm_fold_workspace_bytes(1, Ls)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    p = torch.empty(20, dtype=torch.int32, device="cuda")
    sc = torch.empty(1, device="cuda")
    maps = (C.c_void_p * 1)(S.data_ptr())
    outs = (C.c_void_p * 1)(p.data_ptr())
    st = L.stream_ptr()
    assert L.lib.rnamsm_fold(1, maps, Ls, None, 0, 1.0, 0.0, 3, 0, outs, sc.data_ptr(), ws.data_ptr(), nbytes - 1,
                             st) != 0
    assert b"workspace" in L.lib.rnamsm_last_error()
    assert L.lib.rnamsm_fold(1, maps, Ls, None, 0, 1.0, 0.0, 3, 1, outs, sc.data_ptr(), ws.data_ptr(), nbytes, st) != 0
    assert b"sequences" in L.lib.rnamsm_last_error()
    assert L.lib.rnamsm_fold(1, maps, Ls, None, 2, 1.0, 0.0, 3, 0, outs, sc.data_ptr(), ws.data_ptr(), nbytes, st) != 0
    assert L.lib.rnamsm_fold(1, maps, Ls, None, 0, 0.0, 0.0, 3, 0, outs, sc.data_ptr(), ws.data_ptr(), nbytes, st) != 0
    assert launches() == n0


def test_oversized_request_fails_before_any_launch(pkg):
    S = torch.zeros((1, 1), device="cuda").expand(200_000, 200_000)     # about 320 GB of tables
    n0 = launches()
    with pytest.raises(RuntimeError):
        pkg.fold_pairs(S)
    assert launches() == n0


@pytest.fixture(scope="module")
def model_and_vocab():
    from rnamsm_b200.inference import build_model
    return build_model(None, "cuda", "fp16")


def test_2drb_1_contact_head_and_dca_fold_like_restatement(pkg, msa_2drb_file, model_and_vocab):
    from rnamsm_b200 import fold
    model, vocab = model_and_vocab
    tokens, _ = pkg.ingest_msa(msa_2drb_file, vocab, 512, sys.maxsize, "first")
    seq = fold.query_sequence(tokens, vocab)
    contacts = model.forward_windows(tokens, return_contacts=True)["contacts"]
    out = model(tokens.unsqueeze(0), need_head_weights=True, return_contacts=True, want_logits=False)
    assert torch.equal(contacts, out["contacts"][0])
    pairs, score = pkg.fold_pairs(contacts, seq)
    ref_pairs, ref_score = F.fold(contacts.cpu().numpy(), seq)
    assert np.array_equal(pairs.cpu().numpy(), ref_pairs) and np.float32(score) == ref_score
    all_rows, _ = pkg.ingest_msa(msa_2drb_file, pkg.Vocab(pkg.Alphabet()), sys.maxsize, sys.maxsize, "first")
    dca = pkg.dca_contacts(all_rows)["contacts"]
    pairs, score = pkg.fold_pairs(dca, seq, mode="score")
    ref_pairs, ref_score = F.fold(dca.cpu().numpy(), seq, mode="score")
    assert np.array_equal(pairs.cpu().numpy(), ref_pairs) and np.float32(score) == ref_score
    print(f"2DRB_1 L {len(seq)}: contact head {pkg.dot_bracket(ref_pairs)}")
    print(f"2DRB_1 L {len(seq)}: DCA          {pkg.dot_bracket(pairs)}")


def read_files(prefix):
    from test_fold_cpu import parse_bpseq, parse_ct, parse_dot_bracket
    name, seq, pairs = parse_ct(prefix + ".ct")
    assert parse_bpseq(prefix + ".bpseq") == (seq, pairs)
    head, seq2, db = open(prefix + ".dbn").read().splitlines()
    assert head == ">" + name and seq2 == seq and parse_dot_bracket(db) == pairs
    return seq, pairs


def test_cli_writes_the_api_structure(pkg, msa_2drb_file, model_and_vocab, tmp_path):
    from rnamsm_b200 import fold
    model, vocab = model_and_vocab
    tokens, _ = pkg.ingest_msa(msa_2drb_file, vocab, 512, sys.maxsize, "first")
    seq = fold.query_sequence(tokens, vocab)
    all_rows, _ = pkg.ingest_msa(msa_2drb_file, vocab, sys.maxsize, sys.maxsize, "first")
    dca = pkg.dca_contacts(all_rows)["contacts"]
    head = model.forward_windows(tokens, return_contacts=True)["contacts"]
    np.save(tmp_path / "m.npy", head.cpu().numpy())
    cases = [(["--source", "dca"], dca, dict(mode="score")),
             (["--source", "contact-head"], head, dict(mode="mea")),
             (["--source", "npy", "--map", str(tmp_path / "m.npy"), "--no_canonical", "--min_loop", "0",
               "--gamma", "4"], head, dict(mode="mea", canonical=False, min_loop=0, gamma=4.0)),
             (["--source", "dca", "--mode", "mea", "--threshold", "0.01"], dca, dict(mode="mea", threshold=0.01))]
    for k, (argv, S, kw) in enumerate(cases):
        prefix = str(tmp_path / f"out{k}")
        fold.main(["--MSA_file", msa_2drb_file, "--out_prefix", prefix] + argv)
        got_seq, got_pairs = read_files(prefix)
        assert got_seq == seq
        pairs, _ = pkg.fold_pairs(S, seq, **kw)
        assert got_pairs == pairs.cpu().tolist(), argv
