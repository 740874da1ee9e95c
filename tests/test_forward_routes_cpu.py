"""CPU: the route table, shapes, float64 reference and child plumbing of tests/test_gpu_forward_routes.py
(tests/forward_routes.py)."""
import pytest
import torch

import forward_routes as FR
from oracle import msa_ref as O


@pytest.mark.parametrize("precision", FR.PRECISIONS)
def test_every_threshold_has_a_case_on_each_side(precision):
    """C <= 128 (one-launch row attention), R <= 128 (umma or flash column attention) and R == 1 (column shortcut): the
    values on both sides of each threshold, and both outcomes of each route predicate, appear among the cases."""
    Rs, Cs = {c.R for c in FR.CASES}, {c.C for c in FR.CASES}
    assert {128, 129} <= Cs and {128, 129} <= Rs and {1, 2} <= Rs and 1 in Cs
    for name, pred in FR.THRESHOLDS.items():
        assert {pred(c) for c in FR.CASES} == {True, False}, name
    routes = [FR.routes(c.R, c.C, precision) for c in FR.CASES]
    for key in ("row", "col", "qkv"):
        seen = {r[key] for r in routes}
        if precision in FR.SIXTEEN:
            want = {"row": {"short", "chain"}, "col": {"r1", "umma", "fa"}, "qkv": {"col_major", "token_major"}}[key]
        else:
            want = {"row": {"f32"}, "col": {"r1", "f32"}, "qkv": {"token_major"}}[key]
        assert seen == want, (precision, key, seen)


def test_routes_of_the_issue_table_are_pinned():
    """Each route that no whole-forward test ran before has at least one case here."""
    def cases(pred):
        return [(c.name, p) for c in FR.CASES for p in FR.PRECISIONS if pred(c, p, FR.routes(c.R, c.C, p))]
    assert cases(lambda c, p, r: r["row"] == "chain" and c.R > 128)
    fa = cases(lambda c, p, r: r["col"] == "fa")
    assert len({n.split("-")[0].split("x")[1] for n, _ in fa}) >= 3                 # several C on the flash kernel
    assert cases(lambda c, p, r: r["col"] == "r1" and c.C > 128 and p in FR.SIXTEEN)
    assert cases(lambda c, p, r: p == "tf32x3" and c.C > 128) and cases(lambda c, p, r: p == "tf32x3" and c.R > 128)
    for R, C in ((128, 128), (129, 129), (128, 9), (129, 9), (2, 128), (2, 129)):
        assert f"{R}x{C}" in {n.split("-")[0] for n, _ in cases(lambda c, p, r: True)}
    # every pad layout, and every layout on both sides of the row threshold
    assert {c.pad for c in FR.CASES} == {"none", "cols", "mid", "rows"}
    for pad in ("cols", "mid", "rows"):
        assert {c.C <= 128 for c in FR.CASES if c.pad == pad} == {True, False}, pad
    # the child's list covers every 16-bit route, and forward_batch members sit on both sides of both thresholds
    child = [FR.routes(FR.CASE[n].R, FR.CASE[n].C, "fp16") for n in FR.CHILD_CASES]
    assert {r["row"] for r in child} == {"short", "chain"} and {r["col"] for r in child} == {"r1", "umma", "fa"}
    for members in (FR.BATCH_MEMBERS, FR.CHILD_BATCH):
        assert {m.C <= 128 for m in members} == {True, False} and {m.R <= 128 for m in members} == {True, False}
        assert all(m.R >= 2 for m in members) and any(m.pad == "rows" for m in members)
    assert {128, 129} <= {m.R for m in FR.BATCH_MEMBERS} | {m.C for m in FR.BATCH_MEMBERS}


def test_dense_route_predicate():
    """The tf32 x 3 GEMM needs N % 32 == 0 and K % 32 == 0; every nn.Linear of the model meets it."""
    assert all(FR.dense_route("tf32x3", N, K) == "tf32x3" for N, K in FR.MODEL_GEMMS)
    assert FR.dense_route("tf32x3", 100, 768) == "ffma" and FR.dense_route("tf32x3", 768, 48) == "ffma"
    assert FR.dense_route("fp32", 768, 768) == "ffma" and FR.dense_route("bf16", 768, 768) == "umma16"
    assert FR.routes(300, 33, "tf32x3")["dense"] == "tf32x3"


def test_cases_are_valid_and_tokens_follow_the_layout():
    names = [c.name for c in FR.CASES]
    assert len(set(names)) == len(names) and set(FR.CHILD_CASES) <= set(names)
    sizes = [c.R * c.C for c in FR.CASES]
    assert sizes[-1] == max(sizes)                                    # the largest shape runs last
    for c in FR.CASES + FR.BATCH_MEMBERS + FR.CHILD_BATCH:
        assert c.valid(), c
        t = c.tokens()
        assert t.shape == (1, c.R, c.C) and torch.equal(t, c.tokens())   # seeded
        pad = t[0].eq(O.PAD_IDX)
        row0 = t[0, 0]
        assert row0[0] == O.CLS_IDX and (~pad[0]).sum() >= min(2, c.C)     # row 0 keeps BOS and a residue
        if c.pad == "none":
            assert not pad.any()
        elif c.pad == "cols":
            k = c.pad_cols()
            assert pad[:, c.C - k:].all() and not pad[:, :c.C - k].any()
        elif c.pad == "mid":
            assert pad.sum() == 1 and pad[0, c.C // 2] and 0 < c.C // 2 < c.C - 1
        else:
            k = c.pad_rows()
            assert pad[c.R - k:].all() and not pad[:c.R - k].any()


def test_c1_is_accepted_by_the_forward_entry():
    """C = 1 (BOS only) is a legal grid for rnamsm_msa_forward (it requires R >= 1 and C >= 1), so it is a case."""
    src = open(FR.os.path.join(FR.ROOT, "rna-msm_b200", "csrc", "api.cu")).read()
    assert 'RNAMSM_REQUIRE(R >= 1 && C >= 1, "msa_forward: empty MSA' in src
    assert any(c.C == 1 for c in FR.CASES)


@pytest.mark.parametrize("R,C,pad", [(2, 2, "none"), (3, 6, "mid"), (1, 5, "cols"), (4, 3, "rows")])
def test_float64_reference_agrees_with_the_float32_oracle(R, C, pad):
    case = FR.Case(R, C, pad, 5)
    tokens = case.tokens()
    r64 = FR.reference(tokens)
    r32 = FR.reference(tokens, dtype=torch.float32)
    assert r64["logits"].dtype == torch.float64 and r32["logits"].dtype == torch.float32
    errs = {k: O.rel_err(r32["representations"][k], r64["representations"][k]) for k in (0, 1, FR.LAYERS)}
    errs["logits"] = O.rel_err(r32["logits"], r64["logits"])
    errs["maps"] = O.rel_err(r32["row_attentions"], r64["row_attentions"])
    print(f"[{case.name}] fp32 oracle vs fp64: {errs}")
    assert max(errs.values()) < 2e-6, errs
    assert r64["row_attentions"].shape == (1, FR.LAYERS, FR.H, C, C)
    assert torch.allclose(r64["row_attentions"].sum(-1), torch.ones((), dtype=torch.float64), atol=1e-12)


def test_child_env_replaces_every_switch():
    base = {"PATH": "/bin", "RNAMSM_FUSE_LN": "1", "RNAMSM_PDL": "1", "RNAMSM_ROW_SHORT": "0", "RNAMSM_GEMM_PAIRS": "3"}
    for name, switches in FR.CHILD_ENVS.items():
        env = FR.child_env(name, base)
        assert env["PATH"] == "/bin" and env["RNAMSM_GEMM_PAIRS"] == "3"
        assert {k: env.get(k) for k in FR.SWITCHES} == {k: switches.get(k) for k in FR.SWITCHES}
    assert FR.child_env("default", base).keys().isdisjoint(FR.SWITCHES)
    cmd = FR.child_command("/tmp/x.pt")
    assert cmd[1].endswith("forward_routes.py") and cmd[2] == "/tmp/x.pt"


def test_child_parses_its_arguments_and_stops_at_the_device_check(tmp_path, monkeypatch):
    assert FR.parse_args([str(tmp_path / "o.pt")]).out == str(tmp_path / "o.pt")
    with pytest.raises(SystemExit):
        FR.parse_args([])
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    with pytest.raises(SystemExit, match="no CUDA device"):
        FR.main([str(tmp_path / "o.pt")])
    assert not (tmp_path / "o.pt").exists()
