"""GPU: sequence weights, Neff and mean-field DCA contacts of an alignment (``rnamsm_b200.sequence_weights``,
``rnamsm_b200.dca_contacts``, ``rnamsm_msa_seq_weights``, ``rnamsm_msa_dca``, ``python -m rnamsm_b200.dca``) against the
float64 restatement of tests/dca_ref.py.

The weights are bit-identical (exact integer neighbour counts, one float64 division each), Neff agrees within 1e-12
relative, the contacts within 1e-6 of the restatement's largest entry, and repeated calls give the same bits."""
import sys

import numpy as np
import pytest
import torch

import dca_ref as D

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    import rnamsm_b200
    return rnamsm_b200


def family(N, L, seed, mut=0.15, gap_p=0.05):
    """Seeded alignment with structure: rows are mutated copies of N // 4 + 1 ancestors, so many rows have neighbours
    at the usual thresholds; residues A G C U and the tokens '-', 'X', 'N', <unk>, <mask> (all the gap state)."""
    rng = np.random.default_rng(seed)
    anc = rng.integers(4, 8, size=(N // 4 + 1, L))
    rows = anc[rng.integers(0, anc.shape[0], size=N)]
    hit = rng.random((N, L)) < mut
    rows = np.where(hit, rng.integers(4, 8, size=(N, L)), rows)
    rows = np.where(rng.random((N, L)) < gap_p, rng.choice([10, 8, 9, 3, 11], size=(N, L)), rows)
    t = np.zeros((N, L + 1), dtype=np.int64)
    t[:, 1:] = rows
    return t


def check(pkg, t_np, theta=0.8, lam=0.5, ref=None):
    t = torch.from_numpy(t_np).cuda()
    ref = ref or D.dca(t_np, theta, lam)
    w, neff = pkg.sequence_weights(t, theta)
    out = pkg.dca_contacts(t, theta, lam)
    assert np.array_equal(w.cpu().numpy(), ref["weights"])
    assert torch.equal(out["weights"], w) and out["neff"] == neff
    assert abs(neff - ref["neff"]) <= 1e-12 * ref["neff"]
    c = out["contacts"]
    assert c.dtype == torch.float32 and c.shape == (t_np.shape[1] - 1,) * 2
    got = c.cpu().double().numpy()
    scale = np.abs(ref["contacts"]).max()
    err = np.abs(got - ref["contacts"]).max()
    print(f"[{t_np.shape[0]} x {t_np.shape[1] - 1} theta {theta} lam {lam}] Neff {neff:.4f}; "
          f"max|dc| / max|c_ref| = {err / scale if scale else err:.3e}")
    assert err <= 1e-6 * scale if scale > 0 else not got.any()
    again = pkg.dca_contacts(t, theta, lam)
    assert torch.equal(again["contacts"], c) and torch.equal(again["weights"], w)
    assert np.array_equal(got, got.T) and not np.diag(got).any()
    return out


@pytest.mark.parametrize("N,L", [(1, 1), (1, 50), (7, 1), (300, 129), (5000, 200), (2000, 1100)])
def test_seeded_grids(pkg, N, L):
    check(pkg, family(N, L, N * 7 + L))


def test_2drb_1_all_rows(pkg, msa_2drb_file):
    tokens, _ = pkg.ingest_msa(msa_2drb_file, pkg.Vocab(pkg.Alphabet()), sys.maxsize, sys.maxsize, "first")
    assert tokens.shape[0] == 1176
    out = check(pkg, tokens.cpu().numpy())
    assert 1.0 <= out["neff"] < 1176


@pytest.mark.parametrize("theta", [0.62, 0.8, 1.0])
@pytest.mark.parametrize("lam", [0.1, 0.5])
def test_theta_and_pseudocount(pkg, theta, lam):
    check(pkg, family(300, 129, 21), theta, lam)


def test_ragged_gap_column_identical_rows(pkg):
    """Rows padded at the end, a column of gaps only, and a block of identical rows."""
    t = family(90, 70, 5)
    t[10:20, 1:] = t[10, 1:]
    t[:, 33] = 10
    for r, k in ((3, 5), (40, 20), (41, 69)):
        t[r, 71 - k:] = 1                                                    # <pad>
    out = check(pkg, t)
    w = out["weights"].cpu().numpy()
    assert (w[10:20] <= 0.1).all()


def test_planted_pair_ranks_first(pkg):
    L, i, j = 60, 9, 47
    t = D.planted_alignment(1500, L, i, j, 3, gap_p=0.05)
    c = check(pkg, t)["contacts"].cpu().numpy()
    iu = np.triu_indices(L, 1)
    top = np.argmax(c[iu])
    assert (iu[0][top] + 1, iu[1][top] + 1) == (i, j)


def test_3d_tokens_and_default_arguments(pkg):
    t = torch.from_numpy(family(64, 40, 2)).cuda()
    a = pkg.dca_contacts(t)
    b = pkg.dca_contacts(t.unsqueeze(0), theta=0.8, pseudocount=0.5)
    assert torch.equal(a["contacts"], b["contacts"]) and a["neff"] == b["neff"]
    w, neff = pkg.sequence_weights(t[:, :])
    assert torch.equal(w, a["weights"]) and neff == a["neff"]


def launches(pkg):
    torch.cuda.synchronize()
    return pkg._lib.lib.rnamsm_launch_count()


@pytest.mark.parametrize("L", [1, 16, 17, 100])
def test_launch_counts(pkg, L):
    """Weights: states, neighbour counts, weights + Neff.  DCA: those, single-site, pairs, T diagonal factorisations, T - 1
    panels and T - 1 trailing updates, T - 1 inverse steps, the product, the scores and 3 for APC and
    symmetrisation, T = ceil(4L / 64): 4T + 7."""
    t = torch.from_numpy(family(50, L, L)).cuda()
    pkg.dca_contacts(t)
    n0 = launches(pkg)
    pkg.sequence_weights(t)
    n1 = launches(pkg)
    pkg.dca_contacts(t)
    n2 = launches(pkg)
    T = -(-4 * L // 64)
    assert (n1 - n0, n2 - n1) == (3, 4 * T + 7)


def test_oversized_request_fails_before_any_launch(pkg):
    t = torch.zeros((1, 100_001), dtype=torch.int64, device="cuda")    # two float64 matrices of side 400000: 2.6 TB
    n0 = launches(pkg)
    with pytest.raises(RuntimeError):
        pkg.dca_contacts(t)
    assert launches(pkg) == n0


def test_argument_errors(pkg):
    t = torch.from_numpy(family(8, 6, 1)).cuda()
    n0 = launches(pkg)
    for bad in (t[0], t.unsqueeze(0).expand(2, -1, -1), t.int(), t[:, :1], t[:0]):
        with pytest.raises(ValueError):
            pkg.dca_contacts(bad)
        with pytest.raises(ValueError):
            pkg.sequence_weights(bad)
    for theta in (0.0, 1.5, float("nan")):
        with pytest.raises(ValueError, match="theta"):
            pkg.sequence_weights(t, theta)
        with pytest.raises(ValueError, match="theta"):
            pkg.dca_contacts(t, theta)
    for lam in (0.0, 1.0, -0.5):
        with pytest.raises(ValueError, match="pseudocount"):
            pkg.dca_contacts(t, pseudocount=lam)
    with pytest.raises(RuntimeError, match="CUDA"):
        pkg.dca_contacts(t.cpu())
    L = pkg._lib
    w = torch.empty(8, dtype=torch.float64, device="cuda")
    neff = torch.empty(1, dtype=torch.float64, device="cuda")
    c = torch.empty((6, 6), dtype=torch.float32, device="cuda")
    nbytes = L.lib.rnamsm_dca_workspace_bytes(8, 6)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    st = L.stream_ptr()
    assert L.lib.rnamsm_msa_dca(t.data_ptr(), 8, 7, 0.8, 0.5, w.data_ptr(), neff.data_ptr(), c.data_ptr(),
                                ws.data_ptr(), nbytes - 1, st) != 0
    assert b"workspace" in L.lib.rnamsm_last_error()
    assert L.lib.rnamsm_msa_dca(t.data_ptr(), 8, 7, 0.8, 1.0, w.data_ptr(), neff.data_ptr(), c.data_ptr(),
                                ws.data_ptr(), nbytes, st) != 0
    assert b"pseudocount" in L.lib.rnamsm_last_error()
    assert L.lib.rnamsm_msa_seq_weights(t.data_ptr(), 8, 1, 0.8, w.data_ptr(), neff.data_ptr(), ws.data_ptr(), nbytes,
                                        st) != 0
    assert launches(pkg) == n0


def test_dca_cli(pkg, msa_2drb_file, tmp_path, capsys):
    from rnamsm_b200 import dca
    out, wout = tmp_path / "c.npy", tmp_path / "w.npy"
    dca.main(["--MSA_file", msa_2drb_file, "--out", str(out), "--weights_out", str(wout), "--theta", "0.62"])
    tokens, _ = pkg.ingest_msa(msa_2drb_file, pkg.Vocab(pkg.Alphabet()), sys.maxsize, sys.maxsize, "first")
    ref = pkg.dca_contacts(tokens, theta=0.62)
    c, w = np.load(out), np.load(wout)
    assert c.dtype == np.float32 and np.array_equal(c, ref["contacts"].cpu().numpy())
    assert w.dtype == np.float64 and np.array_equal(w, ref["weights"].cpu().numpy())
    printed = capsys.readouterr().out
    assert f"N {tokens.shape[0]}" in printed and f"L {tokens.shape[1] - 1}" in printed and "Neff" in printed
