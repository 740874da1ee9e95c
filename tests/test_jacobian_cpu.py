"""CPU: the categorical Jacobian -- the float64 contact reference on constructed Jacobians, the substitution list, and
the workspace layouts of rnamsm_jacobian_workspace_bytes / rnamsm_jacobian_contacts_scratch_bytes."""
import ctypes as C

import numpy as np
import pytest

import jacobian_ref as JR


def _planted(P=9, A=4, i=2, j=6, seed=0, scale=1e-3):
    rng = np.random.default_rng(seed)
    J = scale * rng.standard_normal((P, A, P, A))
    block = rng.standard_normal((A, A))
    block = block - block.mean(0) - block.mean(1, keepdims=True) + block.mean()   # survives the centring whole
    J[i, :, j, :] += block
    J[j, :, i, :] += block.T
    return J


# ------------------------------------------------------------------------------------------------ reference
def test_one_axis_terms_centre_to_zero():
    """A J that is a sum of terms each depending on at most three of its four axes has no A x A block left."""
    rng = np.random.default_rng(1)
    P, A = 7, 4
    i, a, j, b = np.ix_(*[np.arange(n) for n in (P, A, P, A)])
    terms = [rng.standard_normal(s) for s in ((P, 1, 1, 1), (1, A, 1, 1), (1, 1, P, 1), (1, 1, 1, A),
                                              (P, A, P, 1), (1, A, P, A), (P, 1, P, A))]
    J = sum(np.broadcast_to(t, (P, A, P, A)) for t in terms)
    assert np.abs(JR.contacts(J)).max() < 1e-12


def test_planted_coupling_is_the_argmax():
    J = _planted()
    c = JR.contacts(J)
    k = np.unravel_index(np.argmax(c), c.shape)
    assert set(k) == {2, 6}


def test_symmetric_with_zero_diagonal():
    J = np.random.default_rng(2).standard_normal((8, 5, 8, 5))
    c = JR.contacts(J)
    assert np.array_equal(c, c.T) and not np.diag(c).any()


def test_equivariant_under_position_permutation():
    J = np.random.default_rng(3).standard_normal((10, 4, 10, 4))
    perm = np.random.default_rng(4).permutation(10)
    Jp = J[perm][:, :, perm]
    assert np.allclose(JR.contacts(Jp), JR.contacts(J)[np.ix_(perm, perm)], rtol=0, atol=1e-12)


def test_zero_total_gives_zeros():
    assert not JR.contacts(np.zeros((5, 4, 5, 4))).any()
    J = np.zeros((5, 4, 5, 4))
    J[:, :, :, 1] = 3.0                                  # a one-axis term only: F is all zero after centring
    assert np.abs(JR.contacts(J)).max() < 1e-12


# ------------------------------------------------------------------------------------------------ substitutions
def test_entries_skip_the_wild_type():
    from rnamsm_b200 import jacobian_entries
    import rnamsm_b200
    v = rnamsm_b200.Vocab(rnamsm_b200.Alphabet()).tokens_to_idx
    alph = [v[c] for c in "AGCU"]
    wt = [v[c] for c in "GAUCN-A"]
    e = jacobian_entries(wt, alph)
    A = len(alph)
    assert e == sorted(set(e))
    assert len(e) == sum(A - (w in alph) for w in wt) == 3 * 5 + 4 * 2
    for s in range(len(wt) * A):
        i, a = divmod(s, A)
        assert (s in e) == (alph[a] != wt[i])
    assert jacobian_entries([v["A"], v["G"]], [v["A"]]) == [1]
    assert jacobian_entries([v["A"]], [v["A"]]) == []


# ------------------------------------------------------------------------------------------------ workspace
def _a(x):
    return (x + 255) // 256 * 256


@pytest.mark.parametrize("R,Cc", [(512, 36), (6, 9), (1, 21), (160, 140)])
@pytest.mark.parametrize("precision", ["fp16", "bf16", "fp32", "tf32x3"])
def test_jacobian_workspace_bytes_matches_layout(R, Cc, precision):
    """The sampling plan of `group` grids with one row, then the wild-type logits [C, D] and the int32 list."""
    from rnamsm_b200 import _lib
    code = _lib.forward_code(precision)
    D = 768
    P, A = Cc - 1, 4
    for g, n in ((1, 3 * P), (3, 3 * P), (14, 4 * P)):
        got = _lib.lib.rnamsm_jacobian_workspace_bytes(R, Cc, D, 12, 3072, code, g, P, A, n)
        sample = _lib.lib.rnamsm_sample_workspace_bytes(R, Cc, D, 12, 3072, code, g, 1)
        assert sample > 0 and got == sample + _a(Cc * D * 4) + _a((1 + P + A + 3 * n) * 4) and got % 256 == 0


def test_jacobian_workspace_bytes_invalid_is_zero():
    from rnamsm_b200 import _lib
    f = _lib.lib.rnamsm_jacobian_workspace_bytes
    assert f(512, 36, 768, 12, 3072, _lib.F16, 1, 35, 4, 105) > 0
    assert f(512, 36, 768, 12, 3072, _lib.F16, 0, 35, 4, 105) == 0
    assert f(512, 36, 768, 12, 3072, _lib.F16, 1, 0, 4, 0) == 0
    assert f(512, 36, 768, 12, 3072, _lib.F16, 1, 35, 0, 0) == 0
    assert f(512, 36, 768, 12, 3072, 7, 1, 35, 4, 105) == 0
    assert b"dtype" in _lib.lib.rnamsm_last_error()


def test_contacts_scratch_bytes():
    from rnamsm_b200 import _lib
    f = _lib.lib.rnamsm_jacobian_contacts_scratch_bytes
    for P, A in ((2, 1), (35, 4), (1023, 4), (100, 7)):
        assert f(P, A) == _a(8 * (P * A) ** 2) + _a(8 * P * P) + _a(8 * (2 * P + 1))
    assert f(0, 4) == 0 and f(4, 0) == 0
