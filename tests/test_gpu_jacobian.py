"""GPU: the categorical Jacobian of the LM head (``MSATransformer.categorical_jacobian``,
``rnamsm_msa_categorical_jacobian``, ``rnamsm_jacobian_contacts``, ``python -m rnamsm_b200.jacobian``).

Every slab of J is bit-identical to the difference of ``forward``'s logits of the substituted grid and of the input,
in every precision and on every route (the batch layer path in groups of grids, one forward per grid); the wild-type
slabs are exactly 0; the contacts follow the float64 restatement of their definition applied to the same J; and J
follows the float64 oracle within the model-level parity bounds of the scoring tests."""
import os

import numpy as np
import pytest
import torch

from oracle import msa_ref as O
import jacobian_ref as JR
import scoring_ref as S

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-4
BF16_TOL = 2e-2
BF16_TOL_DEEP_SHARP = 8e-2


def tol(precision, sharp_deep):
    if precision == "fp32":
        return FP32_TOL
    return BF16_TOL_DEEP_SHARP if sharp_deep else BF16_TOL


@pytest.fixture(scope="module")
def pkg():
    import rnamsm_b200
    return rnamsm_b200


def build(pkg, seed, layers=10, sharpen=1.0, precision="fp32"):
    model = pkg.MSATransformer(pkg.Vocab(pkg.Alphabet()), num_layers=layers, precision=precision)
    sd = O.make_weights(int(seed), num_layers=layers, sharpen=float(sharpen))
    model.load_state_dict(sd, strict=True)
    return model.eval().cuda(), sd


def golden(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    return g, torch.from_numpy(g["tokens"].astype(np.int64))[0]


def alphabet_idx(alphabet):
    return [O.TOK_TO_IDX[c] for c in alphabet]


def forward_jacobian(model, t, row, pos, alph):
    """J from plain forwards: the logits of each substituted grid minus those of t, at (row, pos) x alph."""
    f = lambda g: model(g.unsqueeze(0), want_logits=True)["logits"][0, row][pos][:, alph]
    wt = f(t)
    J = torch.zeros((len(pos), len(alph), len(pos), len(alph)), dtype=torch.float32, device=t.device)
    q = t[row].tolist()
    for i, c in enumerate(pos):
        for a, v in enumerate(alph):
            if q[c] != v:
                g = t.clone()
                g[row, c] = v
                J[i, a] = f(g) - wt
    return J


# ------------------------------------------------------------------------------------------------ bit identity
SHAPES = ["tiny", "tiny_pad", "single_row", "2DRB_1", "seeded_160x140"]


def shape_case(golden_dir, name):
    """-> (weight seed, sharpen, tokens [R, C], [(row, positions)])"""
    if name == "seeded_160x140":
        t = O.make_tokens(160, 140, 11, gap_p=0.1)[0]
        return 11, 1.0, t, [(0, [1, 2, 70, 139]), (97, [5, 64, 65])]
    g, t = golden(golden_dir, name)
    R = t.shape[0]
    if name == "2DRB_1":
        return int(g["wseed"]), float(g["sharpen"]), t, [(0, [1, 2, 17, 35]), (300, [9, 30])]
    cases = [(0, S.default_positions(t, 0)[:6])]
    if R > 2:
        cases.append((R // 2, S.default_positions(t, R // 2)[:4]))
    return int(g["wseed"]), float(g["sharpen"]), t, cases


@pytest.mark.parametrize("name", SHAPES)
@pytest.mark.parametrize("precision", ["fp16", "bf16", "fp32", "tf32x3"])
def test_jacobian_bit_identical_to_forward(pkg, golden_dir, name, precision):
    seed, sharpen, t, cases = shape_case(golden_dir, name)
    model, _ = build(pkg, seed, 10, sharpen, precision)
    t = t.cuda()
    T = t.numel()
    for alphabet in ("AGCU", "U-N"):
        alph = alphabet_idx(alphabet)
        for row, pos in cases:
            ref = forward_jacobian(model, t, row, pos, alph)
            n = len(pkg.jacobian_entries([int(t[row, c]) for c in pos], alph))
            q = t[row].tolist()
            for group in (1, 3, n):                              # the last one runs every substitution in one pass
                c, J = model.categorical_jacobian(t, row=row, positions=pos, alphabet=alphabet, token_budget=group * T,
                                                  return_jacobian=True)
                assert J.shape == (len(pos), len(alph), len(pos), len(alph)) and J.dtype == torch.float32
                assert c.shape == (len(pos), len(pos)) and c.dtype == torch.float32
                assert torch.equal(J, ref), (alphabet, row, group, (J - ref).abs().max().item())
                for i, col in enumerate(pos):
                    for a, v in enumerate(alph):
                        if q[col] == v:
                            assert not J[i, a].any()             # the wild type's slab: exactly 0


def test_default_positions_and_3d_tokens(pkg, golden_dir):
    g, t = golden(golden_dir, "tiny_pad")
    model, _ = build(pkg, g["wseed"], 10, g["sharpen"], "fp16")
    t = t.cuda()
    row = int((t.cpu() == O.PAD_IDX).any(1).nonzero()[0])      # a row with pads
    pos = S.default_positions(t.cpu(), row)
    a, Ja = model.categorical_jacobian(t, row=row, return_jacobian=True)
    b, Jb = model.categorical_jacobian(t.unsqueeze(0), row=row, positions=pos, return_jacobian=True)
    assert a.shape == (len(pos), len(pos)) and torch.equal(a, b) and torch.equal(Ja, Jb)


# ------------------------------------------------------------------------------------------------ contacts
@pytest.mark.parametrize("precision", ["fp16", "fp32"])
def test_contacts_match_reference_and_are_reproducible(pkg, golden_dir, precision):
    g, t = golden(golden_dir, "2DRB_1")
    model, _ = build(pkg, g["wseed"], 10, g["sharpen"], precision)
    t = t[:64].cuda()
    T = t.numel()
    pos = S.default_positions(t.cpu())[:20]
    c, J = model.categorical_jacobian(t, positions=pos, token_budget=4 * T, return_jacobian=True)
    ref = JR.contacts(J.cpu().double().numpy())
    got = c.cpu().double().numpy()
    err = np.linalg.norm(got - ref) / np.linalg.norm(ref)
    print(f"[{precision}] contacts vs float64 restatement on the same J: {err:.3e}")
    assert err <= 1e-5
    assert np.array_equal(got, got.T) and not np.diag(got).any()
    c2, J2 = model.categorical_jacobian(t, positions=pos, token_budget=4 * T, return_jacobian=True)
    c3, J3 = model.categorical_jacobian(t, positions=pos, token_budget=11 * T, return_jacobian=True)
    assert torch.equal(c, c2) and torch.equal(c, c3) and torch.equal(J, J2) and torch.equal(J, J3)


def test_contacts_entry_on_constructed_jacobians(pkg):
    """rnamsm_jacobian_contacts alone: a planted coupling comes out on top, and a J without any A x A structure gives
    zeros (total == 0)."""
    L = pkg._lib

    def run(J):
        J = torch.from_numpy(np.ascontiguousarray(J, dtype=np.float32)).cuda()
        P, A = J.shape[:2]
        out = torch.full((P, P), float("nan"), device="cuda")
        nbytes = L.lib.rnamsm_jacobian_contacts_scratch_bytes(P, A)
        scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        L.check(L.lib.rnamsm_jacobian_contacts(J.data_ptr(), P, A, out.data_ptr(), scratch.data_ptr(), nbytes,
                                               L.stream_ptr()), "jacobian_contacts")
        return out.cpu().double().numpy()

    rng = np.random.default_rng(0)
    P, A = 30, 4
    J = 1e-3 * rng.standard_normal((P, A, P, A))
    J[3, :, 17, :] += rng.standard_normal((A, A))
    J[17, :, 3, :] += rng.standard_normal((A, A))
    got = run(J)
    ref = JR.contacts(J.astype(np.float32))
    assert np.linalg.norm(got - ref) / np.linalg.norm(ref) <= 1e-5
    assert set(np.unravel_index(np.argmax(got), got.shape)) == {3, 17}
    assert not run(np.zeros((5, 4, 5, 4))).any()


# ------------------------------------------------------------------------------------------------ float64 oracle
@pytest.mark.parametrize("name", ["tiny", "tiny_pad"])
@pytest.mark.parametrize("precision", ["fp32", "fp16", "bf16"])
def test_jacobian_vs_float64_oracle(pkg, golden_dir, name, precision):
    g, t = golden(golden_dir, name)
    layers, sharpen = int(g["layers"]), float(g["sharpen"])
    model, sd = build(pkg, g["wseed"], layers, sharpen, precision)
    pos = S.default_positions(t)[:5]
    alph = alphabet_idx("AGCU")
    ref = JR.jacobian(O.to_dtype(sd, torch.float64), t, pos, alph)
    J = model.categorical_jacobian(t.cuda(), positions=pos, return_jacobian=True)[1].cpu().double().numpy()
    err = np.abs(J - ref).max() / np.abs(ref).max()
    print(f"[{name}/{precision}] max|dJ| / max|J_ref| = {err:.3e}")
    assert err <= tol(precision, sharpen >= 3 and layers >= 10)


# ------------------------------------------------------------------------------------------------ routing
def launches(pkg):
    return pkg._lib.lib.rnamsm_launch_count()


def test_routing_launch_counts(pkg):
    """16-bit: the wild-type run is rnamsm_msa_forward_batch on one grid minus its final LayerNorm, plus 5 launches
    (row gather, final LayerNorm, LM-head dense, LM-head LayerNorm, vocab projection); a pass of g grids is
    rnamsm_msa_forward_batch on g grids minus its final LayerNorm, plus 7 (variant grids and collect besides those
    five); the contacts are 8.  fp32: one forward per grid without its final LayerNorm, and the same counts around it."""
    t = O.make_tokens(24, 30, 3, pad_cols=2)[0]
    t[0, 1:4] = torch.tensor(alphabet_idx("AGC"))            # 3 substitutions each: 9 grids, three passes of 3
    t = t.cuda()
    T = t.numel()
    pos = [1, 2, 3]
    grids = [t.clone() for _ in range(3)]
    m16, _ = build(pkg, 4, 3, 1.0, "fp16")
    m16.categorical_jacobian(t, positions=pos, token_budget=3 * T)      # warm: weights staged, modules loaded
    torch.cuda.synchronize()
    c0 = launches(pkg)
    m16.forward_batch([t])
    c1 = launches(pkg)
    m16.forward_batch(grids)
    c2 = launches(pkg)
    m16.categorical_jacobian(t, positions=pos, token_budget=3 * T)
    c3 = launches(pkg)
    b1, b3 = c1 - c0, c2 - c1
    assert c3 - c2 == (b1 - 1 + 5) + 3 * (b3 - 1 + 7) + 8
    m32, _ = build(pkg, 4, 3, 1.0, "fp32")
    m32(t.unsqueeze(0), want_logits=False)
    c0 = launches(pkg)
    m32(t.unsqueeze(0), want_logits=False)
    c1 = launches(pkg)
    m32.categorical_jacobian(t, positions=pos, token_budget=3 * T)
    c2 = launches(pkg)
    f = c1 - c0
    assert c2 - c1 == (f - 1 + 5) + 3 * (3 * (f - 1) + 7) + 8


# ------------------------------------------------------------------------------------------------ arguments
def test_argument_errors(pkg, golden_dir):
    g, t = golden(golden_dir, "tiny_pad")
    model, _ = build(pkg, g["wseed"], 2, 1.0, "fp16")
    t = t.cuda()
    R, Cc = t.shape
    prow = int((t.cpu() == O.PAD_IDX).any(1).nonzero()[0])
    pcol = int((t[prow].cpu() == O.PAD_IDX).nonzero()[0])
    for alphabet, match in (("", "empty"), ("AGA", "repeats"), ("AGT", "residue or gap"), ("A<mask>", "residue or gap")):
        with pytest.raises(ValueError, match=match):
            model.categorical_jacobian(t, alphabet=alphabet)
    with pytest.raises(ValueError, match="outside"):
        model.categorical_jacobian(t, positions=[1, Cc])
    with pytest.raises(ValueError, match="outside"):
        model.categorical_jacobian(t, positions=[-1, 2])
    with pytest.raises(ValueError, match="BOS"):
        model.categorical_jacobian(t, positions=[0, 2])
    with pytest.raises(ValueError, match="padding"):
        model.categorical_jacobian(t, row=prow, positions=[1, pcol])
    with pytest.raises(ValueError, match="row"):
        model.categorical_jacobian(t, row=R)
    with pytest.raises(ValueError, match="two positions"):
        model.categorical_jacobian(t, positions=[3])
    with pytest.raises(RuntimeError, match="CUDA"):
        model.categorical_jacobian(t.cpu())


# ------------------------------------------------------------------------------------------------ CLI
def test_jacobian_cli(pkg, msa_2drb_file, tmp_path):
    from rnamsm_b200 import jacobian
    out, jout = tmp_path / "contacts.npy", tmp_path / "J.npy"
    jacobian.main(["--MSA_file", msa_2drb_file, "--out", str(out), "--jacobian_out", str(jout),
                   "--max_seqs_per_msa", "8"])
    c, J = np.load(out), np.load(jout)
    L_ = c.shape[0]
    assert c.shape == (L_, L_) and c.dtype == np.float32 and L_ > 2
    assert J.shape == (L_, 4, L_, 4) and J.dtype == np.float32
    assert np.isfinite(c).all() and np.array_equal(c, c.T) and not np.diag(c).any()
