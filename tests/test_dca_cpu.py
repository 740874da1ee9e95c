"""CPU: the float64 restatement of the alignment statistics (tests/dca_ref.py) on constructed alignments, and the
argument parsing of ``python -m rnamsm_b200.dca``."""
import numpy as np
import pytest

import dca_ref as D


def grid(rows):
    """residue strings -> int64 tokens [N, L + 1] with BOS"""
    idx = {"A": 4, "G": 5, "C": 6, "U": 7, "X": 8, "N": 9, "-": 10}
    return np.array([[0] + [idx[c] for c in r] for r in rows], dtype=np.int64)


def random_grid(N, L, seed):
    rng = np.random.default_rng(seed)
    t = np.zeros((N, L + 1), dtype=np.int64)
    t[:, 1:] = rng.integers(4, 11, size=(N, L))
    return t


def test_states_map_residues_and_gap_state():
    t = np.array([[0, 4, 5, 6, 7, 8, 9, 10, 1, 3, 11]])
    assert D.states(t).tolist() == [[0, 1, 2, 3, 4, 4, 4, 4, 4, 4]]
    assert D.states(t[None]).tolist() == D.states(t).tolist()


def test_distinct_rows_have_unit_weights():
    t = grid(["AAAAA", "GGGGG", "CCCCC", "UUUUU", "-----"])
    w, neff = D.weights(t)
    assert w.tolist() == [1.0] * 5 and neff == 5.0


def test_duplicate_rows_share_their_weight():
    rows = ["ACGUACGUAC"] * 3 + ["GGGGGCCCCC"] * 2 + ["UUUUUAAAAA"]
    w, neff = D.weights(grid(rows))
    assert w.tolist() == [1 / 3] * 3 + [0.5] * 2 + [1.0]
    assert neff == pytest.approx(3.0, abs=1e-15)


@pytest.mark.parametrize("mismatches,neighbours", [(1, True), (2, True), (3, False)])
def test_identity_boundary(mismatches, neighbours):
    """L = 10, theta = 0.8: 8 matches (2 mismatches) make a neighbour, 7 do not; gap == gap is a match."""
    a = "ACGU-ACGU-"
    b = "".join(("G" if c != "G" else "A") if k < mismatches else c for k, c in enumerate(a))
    w, _ = D.weights(grid([a, b]), 0.8)
    assert w.tolist() == ([0.5, 0.5] if neighbours else [1.0, 1.0])


def test_theta_one_needs_identical_rows():
    w, _ = D.weights(grid(["ACGUA", "ACGUA", "ACGUC"]), 1.0)
    assert w.tolist() == [0.5, 0.5, 1.0]


@pytest.mark.parametrize("lam", [0.1, 0.5])
def test_covariance_is_symmetric_positive_definite(lam):
    C, _, _ = D.covariance(random_grid(60, 12, 3), 0.8, lam)
    assert C.shape == (48, 48)
    assert np.array_equal(C, C.T)
    np.linalg.cholesky(C)
    assert np.linalg.eigvalsh(C).min() > 0


@pytest.mark.parametrize("seed", [1, 2])
def test_planted_pair_ranks_first(seed):
    L, i, j = 30, 6, 21
    t = D.planted_alignment(400, L, i, j, seed, gap_p=0.05)
    c = D.dca(t)["contacts"]
    assert np.allclose(c, c.T) and not np.diag(c).any()
    iu = np.triu_indices(L, 1)
    top = np.argmax(c[iu])
    assert (iu[0][top] + 1, iu[1][top] + 1) == (i, j)


def test_single_column_and_single_row():
    r = D.dca(grid(["A"]))
    assert r["contacts"].shape == (1, 1) and r["contacts"][0, 0] == 0.0 and r["neff"] == 1.0
    r = D.dca(grid(["ACGUACGU"]), 0.8, 0.1)
    assert r["contacts"].shape == (8, 8) and np.isfinite(r["contacts"]).all()


def test_cli_parses_arguments():
    from rnamsm_b200 import dca
    a = dca.parse_args(["--MSA_file", "x.a2m_msa2", "--out", "c.npy"])
    assert (a.MSA_file, a.out, a.theta, a.pseudocount, a.weights_out) == ("x.a2m_msa2", "c.npy", 0.8, 0.5, None)
    a = dca.parse_args(["--MSA_file", "x", "--out", "c.npy", "--theta", "0.62", "--pseudocount", "0.1",
                        "--weights_out", "w.npy"])
    assert (a.theta, a.pseudocount, a.weights_out) == (0.62, 0.1, "w.npy")
    with pytest.raises(SystemExit):
        dca.parse_args(["--out", "c.npy"])


def test_python_argument_errors_before_the_device():
    """Shape, theta and pseudocount are checked before anything touches a device; CPU tensors are refused."""
    import torch
    from rnamsm_b200 import coevolution as CO
    t = torch.zeros((3, 5), dtype=torch.int64)
    for bad, match in ((torch.zeros((2, 3, 5), dtype=torch.int64), "expected"), (torch.zeros(5, dtype=torch.int64), "expected"),
                       (t.int(), "int64"), (torch.zeros((0, 5), dtype=torch.int64), "at least"),
                       (torch.zeros((3, 1), dtype=torch.int64), "at least")):
        with pytest.raises(ValueError, match=match):
            CO.dca_contacts(bad)
    for theta in (0.0, -0.1, 1.01, float("nan")):
        with pytest.raises(ValueError, match="theta"):
            CO.sequence_weights(t, theta=theta)
    for lam in (0.0, 1.0, float("nan")):
        with pytest.raises(ValueError, match="pseudocount"):
            CO.dca_contacts(t, pseudocount=lam)
    with pytest.raises(RuntimeError, match="CUDA"):
        CO.sequence_weights(t)
    with pytest.raises(RuntimeError, match="CUDA"):
        CO.dca_contacts(t)


def test_workspace_sizes_are_host_math():
    from rnamsm_b200 import _lib as L
    assert L.lib.rnamsm_seq_weights_workspace_bytes(0, 10) == 0
    assert L.lib.rnamsm_dca_workspace_bytes(10, 0) == 0
    a = L.lib.rnamsm_dca_workspace_bytes(100, 100)
    mp = 448                                                     # 4 * 100 rounded up to a multiple of 64
    assert a % 256 == 0 and 2 * mp * mp * 8 < a < 2 * mp * mp * 8 + 2 ** 20
    assert L.lib.rnamsm_seq_weights_workspace_bytes(10 ** 5, 200) < 2 * 10 ** 7
