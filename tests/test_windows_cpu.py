"""CPU: full-length features from overlapping windows -- rnamsm_window_starts against the restatement in
windows_ref.py, the stitching coefficients, the workspace layout of rnamsm_windows_workspace_bytes, and the argument
handling of the inference CLI."""
import ctypes as C

import numpy as np
import pytest

import windows_ref as WR


def lib_starts(L, window, stride):
    from rnamsm_b200 import _lib
    K = _lib.lib.rnamsm_window_starts(L, window, stride, None)
    if K == 0:
        return None
    out = (C.c_int * K)()
    assert _lib.lib.rnamsm_window_starts(L, window, stride, out) == K
    return list(out)


# ------------------------------------------------------------------------------------------------ plan
GRID = [(L, w, s) for L in (1, 2, 5, 63, 64, 100, 150, 1023, 1024, 1501, 3000)
        for w in (1, 7, 63, 64, 1023) for s in sorted({1, 2, max(1, w // 2), max(1, w - 1), w}) if s <= w]


@pytest.mark.parametrize("L,window,stride", GRID)
def test_window_starts_match_restatement(L, window, stride):
    got = lib_starts(L, window, stride)
    ref = WR.window_starts(L, window, stride)
    assert got == ref
    W = min(window, L)
    assert got[0] == 0 and got[-1] == L - W                          # the last window ends at the last residue
    assert all(b > a for a, b in zip(got, got[1:]))                   # strictly ascending
    assert all(b - a <= stride for a, b in zip(got, got[1:]))         # no residue is left out
    if L <= window:
        assert got == [0]


def test_window_starts_special_cases():
    assert lib_starts(100, 64, 64) == [0, 36]                          # stride == window: the last window is end-aligned
    assert lib_starts(128, 64, 64) == [0, 64]                          # no overlap at all
    assert lib_starts(70, 64, 1) == list(range(7))                    # stride 1: every offset
    assert lib_starts(1501, 1023, 511) == [0, 478]
    assert lib_starts(3000, 1023, 511) == [0, 511, 1022, 1533, 1977]


@pytest.mark.parametrize("L,window,stride,match", [(0, 64, 32, "residue"), (-3, 64, 32, "residue"),
                                                   (100, 64, 0, "stride"), (100, 64, 65, "stride"),
                                                   (100, 0, 0, "stride"), (100, 64, -1, "stride")])
def test_window_starts_invalid_is_zero(L, window, stride, match):
    from rnamsm_b200 import _lib
    assert _lib.lib.rnamsm_window_starts(L, window, stride, None) == 0
    assert match.encode() in _lib.lib.rnamsm_last_error()
    assert WR.window_starts(L, window, stride) is None


# ------------------------------------------------------------------------------------------------ coefficients
@pytest.mark.parametrize("L,window,stride", [(150, 64, 32), (150, 64, 64), (150, 64, 1), (100, 64, 20), (60, 64, 32),
                                             (1501, 1023, 511), (200, 50, 17)])
def test_coefficients_sum_to_one(L, window, stride):
    starts = WR.window_starts(L, window, stride)
    W = min(window, L)
    c1, c2 = WR.coefficients(L, W, starts)
    assert np.abs(c1.sum(0) - 1).max() < 1e-12                          # every residue is covered
    cov = WR.covered(L, W, starts)
    s = c2.sum(0)
    assert np.abs(s[cov] - 1).max() < 1e-12
    assert not s[~cov].any()
    one = WR.single(L, W, starts)
    k, i, j = one[one >= 0], *np.nonzero(one >= 0)
    assert (c2[k, i, j] == 1.0).all()                                 # a pair one window holds takes its value as is
    if L <= window:
        assert cov.all() and (one == 0).all()


def test_tent_weights_favour_the_window_centre():
    W, s = 64, 10
    w = WR.tent(np.arange(s, s + W), s, W)
    assert w[0] == 1 and w[-1] == 1 and w.max() == W // 2 and (w >= 1).all()
    assert (w == w[::-1]).all()


def test_stitch_restatement_on_constant_windows():
    """Windows that agree where they overlap stitch to that common value; disjoint pairs are 0."""
    rng = np.random.default_rng(0)
    L, window, stride, D, NH = 150, 64, 32, 5, 3
    starts = WR.window_starts(L, window, stride)
    full_emb, full_map = rng.standard_normal((L, D)), rng.standard_normal((NH, L, L))
    W = window
    embs = np.stack([full_emb[s:s + W] for s in starts])
    maps = np.stack([full_map[:, s:s + W, s:s + W] for s in starts])
    emb, atp, con = WR.stitch(embs, maps, starts, L, contacts=maps[:, 0])
    cov = WR.covered(L, W, starts)
    assert np.allclose(emb, full_emb, rtol=0, atol=1e-12)
    assert np.allclose(atp[:, cov], full_map[:, cov], rtol=0, atol=1e-12) and not atp[:, ~cov].any()
    assert np.allclose(con[cov], full_map[0][cov], rtol=0, atol=1e-12)


# ------------------------------------------------------------------------------------------------ workspace
def _a(x):
    return (x + 255) // 256 * 256


@pytest.mark.parametrize("R,Cc,window,stride", [(32, 1502, 1023, 511), (128, 1502, 1023, 511), (6, 151, 63, 31),
                                                (1, 151, 63, 31), (4, 40, 63, 31)])
@pytest.mark.parametrize("precision", ["fp16", "bf16", "fp32", "tf32x3"])
@pytest.mark.parametrize("contacts", [0, 1])
def test_windows_workspace_bytes_matches_layout(R, Cc, window, stride, precision, contacts):
    """tok | x | forward workspace | maps | row 0 (R >= 2) | contacts and their scratch | starts, for min(group, K)."""
    from rnamsm_b200 import _lib
    code = _lib.forward_code(precision)
    D, H, F, N = 768, 12, 3072, 10
    NH = N * H
    starts = WR.window_starts(Cc - 1, window, stride)
    K, W = len(starts), min(window, Cc - 1)
    Cw, T = W + 1, R * (W + 1)
    for group in (1, 2, 100):
        g = min(group, K)
        if precision in ("fp16", "bf16") and R >= 2:
            fwd = _lib.lib.rnamsm_batch_workspace_bytes(g, (C.c_int * g)(*[R] * g), (C.c_int * g)(*[Cw] * g), D, H, F, code)
        else:
            fwd = _lib.lib.rnamsm_workspace_bytes(R, Cw, D, H, F, code) + _a(T)
        assert fwd > 0
        want = (_a(g * T * 8) + _a(g * T * D * 4) + _a(fwd) + _a(g * NH * Cw * Cw * 4) + (_a(g * Cw * D * 4) if R > 1 else 0)
                + (_a(g * W * W * 4) + _a(NH * Cw * 4) if contacts else 0) + _a((K + 1) * 4))
        got = _lib.lib.rnamsm_windows_workspace_bytes(R, Cc, D, H, F, N, code, group, window, stride, contacts)
        assert got == want and got % 256 == 0


def test_windows_workspace_bytes_invalid_is_zero():
    from rnamsm_b200 import _lib
    f = _lib.lib.rnamsm_windows_workspace_bytes
    assert f(32, 1502, 768, 12, 3072, 10, _lib.F16, 1, 1023, 511, 0) > 0
    assert f(32, 1502, 768, 12, 3072, 10, _lib.F16, 0, 1023, 511, 0) == 0
    assert f(32, 1, 768, 12, 3072, 10, _lib.F16, 1, 1023, 511, 0) == 0
    assert f(32, 1502, 768, 12, 3072, 0, _lib.F16, 1, 1023, 511, 0) == 0
    assert f(32, 1502, 768, 12, 3072, 10, _lib.F16, 1, 1023, 0, 0) == 0
    assert b"stride" in _lib.lib.rnamsm_last_error()
    assert f(32, 1502, 768, 12, 3072, 10, 7, 1, 1023, 511, 0) == 0
    assert b"dtype" in _lib.lib.rnamsm_last_error()


# ------------------------------------------------------------------------------------------------ CLI
def test_cli_defaults_keep_the_crop():
    from rnamsm_b200 import inference
    a = inference.parse_args([])
    assert a.long == "crop" and a.window is None and a.stride is None


def test_cli_window_flags():
    from rnamsm_b200 import inference
    a = inference.parse_args(["--long", "window", "--window", "512", "--stride", "128"])
    assert (a.long, a.window, a.stride) == ("window", 512, 128)
    a = inference.parse_args(["--long", "window"])
    assert (a.long, a.window, a.stride) == ("window", None, None)


@pytest.mark.parametrize("argv", [["--long", "tile"], ["--window", "512"], ["--stride", "8"],
                                  ["--long", "crop", "--window", "512"], ["--long", "window", "--window", "0"],
                                  ["--long", "window", "--stride", "-2"], ["--long", "window", "--window", "x"]])
def test_cli_rejects_bad_flags(argv, capsys):
    from rnamsm_b200 import inference
    with pytest.raises(SystemExit) as e:
        inference.parse_args(argv)
    assert e.value.code == 2
