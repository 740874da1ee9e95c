"""CPU checks of tests/rowwise_cases.py: the LayerNorm gate holds for an fp32 emulation of warp_layernorm in every
regime, width and output type, and rejects a one-pass variance; the exact-operand builders are exact; the float64
references agree with the oracle (oracle/msa_ref.py).  (The GPU side is tests/test_gpu_rowwise_edges.py.)"""
import numpy as np
import pytest
import torch

import rowwise_cases as RC
from oracle import msa_ref as O

WIDTHS = [128 * k for k in range(1, 9)]


def emulated(x, w, b, code, ulps=0, one_pass=False):
    return RC.round_out(torch.from_numpy(RC.emulate_layernorm(x, w, b, rsqrt_ulps=ulps, one_pass=one_pass)), code)


@pytest.mark.parametrize("D", WIDTHS)
def test_gate_holds_for_emulation(D):
    """Every regime, rsqrtf at -2, 0 and +2 ulp, all three output types, normal and saturating weights.  The worst
    ratio of error to gate is printed (run with -s).  fp32 outputs must stay below 1/2 of the gate.  A 16-bit output's
    own rounding (half an ulp) is reached by construction, so there the ratio only has to stay below 1."""
    worst = {}
    for saturating in (False, True):
        w, b = RC.ln_affine(D, 5, saturating)
        for regime in RC.ROW_REGIMES:
            x = RC.ln_rows(regime, 24, D, seed=3)
            for code in (0, 1, 2):
                ref, gate = RC.ln_reference(torch.from_numpy(x), torch.from_numpy(w), torch.from_numpy(b), code)
                for ulps in (-2, 0, 2):
                    got = emulated(x, w, b, code, ulps)
                    assert bool(torch.isfinite(got.float()).all())
                    key = (regime, code, saturating)
                    worst[key] = max(worst.get(key, 0.0), RC.gate_ratio(got, ref, gate))
    for code, limit in ((0, 0.5), (1, 1.0), (2, 1.0)):
        k, v = max(((k, v) for k, v in worst.items() if k[1] == code), key=lambda kv: kv[1])
        print(f"D={D} out {code}: worst gate ratio {v:.3f} at {k}")
        assert v < limit, worst


@pytest.mark.parametrize("D", [128, 768, 1024])
def test_gate_rejects_one_pass_variance(D):
    """E[x^2] - mu^2 fails the gate on `offset` rows at every output type; on randn rows it passes (the existing
    tests' rows cannot tell the two apart)."""
    w, b = RC.ln_affine(D, 5)
    wt, bt = torch.from_numpy(w), torch.from_numpy(b)
    for code in (0, 1, 2):
        x = RC.ln_rows("offset", 24, D, seed=3)
        ref, gate = RC.ln_reference(torch.from_numpy(x), wt, bt, code)
        assert RC.gate_ratio(emulated(x, w, b, code, one_pass=True), ref, gate) > 10.0
        x = RC.ln_rows("randn", 24, D, seed=3)
        ref, gate = RC.ln_reference(torch.from_numpy(x), wt, bt, code)
        assert RC.gate_ratio(emulated(x, w, b, code, one_pass=True), ref, gate) < 1.0


@pytest.mark.parametrize("D", WIDTHS)
def test_exact_b_regimes(D):
    """constant_grid rows: every fp32 partial sum is exact (so the row mean is the value itself); with zero rows, the
    emulated output is exactly b rounded once to the output type."""
    x = RC.ln_rows("constant_grid", 16, D, seed=3)
    c = x[:, :1].astype(np.float64)
    assert np.array_equal(np.cumsum(x, axis=1, dtype=np.float32), np.cumsum(x, axis=1, dtype=np.float64))
    assert np.array_equal(x.sum(1, dtype=np.float32) / np.float32(D), c[:, 0].astype(np.float32))
    w, b = RC.ln_affine(D, 5)
    for regime in RC.EXACT_B_REGIMES:
        x = RC.ln_rows(regime, 16, D, seed=3)
        for code in (0, 1, 2):
            want = RC.ln_expected_b(torch.from_numpy(b), code).expand(16, D)
            assert torch.equal(emulated(x, w, b, code), want)


def test_regimes_have_their_shape():
    D = 768
    x = RC.ln_rows("offset", 8, D, 1).astype(np.float64)
    assert np.all(np.abs(x.mean(1) / x.std(1)) > 5e3)
    x = RC.ln_rows("outlier", 8, D, 1)
    assert np.all(np.abs(x[:, RC.outlier_features(D)]) == 1e3)
    x = RC.ln_rows("near_eps", 8, D, 1).astype(np.float64)
    assert np.all((x.var(1) > 1e-7) & (x.var(1) < 1e-5))
    w, _ = RC.ln_affine(D, 5, saturating=True)
    ref, _ = RC.ln_reference(torch.from_numpy(RC.ln_rows("randn", 8, D, 1)), torch.from_numpy(w), torch.zeros(D), 0)
    assert float(ref.abs().max()) > 1.5 * RC.F16_MAX


def test_mixed_rows_cover_every_regime():
    x, reg = RC.ln_mixed_rows(23, 256, seed=1, rotate=3)
    assert set(reg.tolist()) == set(range(len(RC.ROW_REGIMES)))
    for k, name in enumerate(RC.ROW_REGIMES):
        assert np.array_equal(x[reg == k], RC.ln_rows(name, int((reg == k).sum()), 256, 1))


def test_ln_reference_matches_oracle():
    x = torch.randn(9, 768, generator=torch.Generator().manual_seed(1), dtype=torch.float64) * 3 + 0.5
    w = 1 + 0.1 * torch.randn(768, dtype=torch.float64)
    b = 0.1 * torch.randn(768, dtype=torch.float64)
    ref, _ = RC.ln_reference(x, w, b, 0, eps=O.LN_EPS)
    assert torch.allclose(ref, O.layer_norm(x, w, b), rtol=0, atol=1e-12)


def test_embed_reference_matches_oracle():
    R, C = 5, 70
    sd = O.make_weights(3, num_layers=1)
    tokens = RC.embed_tokens(R, C, O.VOCAB, O.PAD_IDX, seed=2)
    ref_o, pm = O.embed({k: v.double() for k, v in sd.items()}, tokens[None])
    ref, _, pad = RC.embed_reference(tokens, sd["embed_tokens.weight"], sd["embed_positions.weight"],
                                     sd["msa_position_embedding"].reshape(-1), sd["emb_layer_norm_before.weight"],
                                     sd["emb_layer_norm_before.bias"], O.PAD_IDX, eps=O.LN_EPS)
    assert torch.equal(pad, pm[0])
    assert torch.allclose(ref, ref_o[0], rtol=0, atol=1e-12)
    assert torch.equal(RC.positions(tokens, O.PAD_IDX), O.positions_from_tokens(tokens))


def test_embed_tokens_layout():
    R, C, V, P = 4, 130, 12, 1
    t = RC.embed_tokens(R, C, V, P, seed=0)
    pos = RC.positions(t, P)
    assert int(pos.max()) == int(pos[0, -1]) == C + P            # row 0 holds the table's last row
    for c in (31, 32, 63, 64, 127):
        assert int(t[1, c]) == P
    assert int(t[1, 33]) != P and int(t[1, 65]) != P and int(t[1, 128]) != P
    assert int(t[2, 0]) == 0 and bool(t[2, 1:].eq(P).all())
    assert {0, V - 1} <= set(t.unique().tolist())


def test_embed_tables_sum_exactly():
    tok, pos, row = RC.embed_tables(12, 40, 6, 256, seed=1, pad_idx=1)
    s32 = (tok[:, None, None, :] + pos[None, :, None, :]).astype(np.float32) + row[None, None, :, None]
    s64 = tok[:, None, None, :].astype(np.float64) + pos[None, :, None, :] + row[None, None, :, None]
    assert np.array_equal(s32.astype(np.float32).astype(np.float64), s64)


@pytest.mark.parametrize("D", [128, 1024])
def test_vocab_exact_operands_are_exact(D):
    h, E, b = RC.vocab_exact_operands(64, 32, D, seed=1)
    ref, _ = RC.vocab_reference(torch.from_numpy(h), torch.from_numpy(E), torch.from_numpy(b))
    # each lane's partial sums, every butterfly partial and the result stay on the 2^-10 grid below 2^14
    prods = h.astype(np.float64)[:, None, :] * E.astype(np.float64)[None, :, :]
    assert np.all(prods * 1024 == np.round(prods * 1024))
    assert float(np.abs(prods).sum(-1).max()) + 1 < 2 ** 14
    acc32 = np.zeros((64, 32), dtype=np.float32)
    for k in range(D):
        acc32 = (acc32 + (h[:, None, k] * E[None, :, k]).astype(np.float32)).astype(np.float32)
    assert np.array_equal((acc32 + b).astype(np.float64), ref.numpy())


def test_vocab_gate_holds_for_fp32():
    h = torch.randn(50, 768, generator=torch.Generator().manual_seed(2))
    E, b = torch.randn(12, 768), torch.randn(12)
    ref, gate = RC.vocab_reference(h, E, b)
    assert RC.gate_ratio(h @ E.T + b, ref, gate) < 0.5


@pytest.mark.parametrize("kind", RC.CONTACT_MAPS)
def test_contact_reference_matches_oracle(kind):
    K, C = 24, 33
    maps = torch.from_numpy(RC.contact_maps(kind, K, C, seed=1)).double()
    w, b = torch.randn(K, dtype=torch.float64), torch.randn(1, dtype=torch.float64)
    out, logit, gate = RC.contact_reference(maps, 1, C - 1, w, b)
    sd = {"contact_head.regression.weight": w.view(1, K), "contact_head.regression.bias": b}
    ref = O.contact_head(sd, None, maps.view(1, 2, 12, C, C))[0]
    assert torch.equal(torch.isnan(out), torch.isnan(ref))
    assert bool(torch.isnan(out).all()) == (kind == "all_bos")
    ok = ~torch.isnan(ref)
    assert torch.allclose(out[ok], ref[ok], rtol=0, atol=1e-12)
    assert bool((gate[ok] > 0).all())


def test_contact_maps_have_their_shape():
    K, C = 4, 40
    A = {k: RC.contact_maps(k, K, C, 1).astype(np.float64) for k in RC.CONTACT_MAPS}
    for k, a in A.items():
        assert np.all(a >= 0) and np.allclose(a.sum(-1), 1.0, atol=1e-5), k
    col = A["column"].sum(-2)
    assert np.all(col.max(-1) > 10 * np.median(col, -1))
    assert np.all(np.triu(A["asymmetric"][:, 1:, 1:]) == 0)
    assert np.all(A["sink"][:, 1:, 1:].sum((-1, -2)) < 2e-3 * C)
    assert np.all(A["all_bos"][:, :, 1:] == 0)


@pytest.mark.parametrize("code", [1, 2], ids=["bf16", "f16"])
def test_range_reference(code):
    dt = torch.float16 if code == 2 else torch.bfloat16
    buf = RC.range_buffer(code, 5000, seed=1)
    count, bits = RC.range_reference(buf, code)
    v = torch.from_numpy(buf.view(np.int16)).view(dt).float()
    edge_val = 65504.0 if code == 2 else float(torch.finfo(torch.bfloat16).max)
    want_count = int((~torch.isfinite(v) | (v.abs() == edge_val)).sum())
    assert count == want_count == 3 * 10           # 5 edge words of each sign, each placed three times
    finite = v[torch.isfinite(v) & (v.abs() != edge_val)]
    want_max = float(finite.abs().max())
    assert bits == int(np.array([want_max], dtype=np.float32).view(np.uint32)[0])
    assert RC.range_reference(np.zeros(0, np.uint16), code) == (0, 0)
    tiny = RC.range_patterns(code)[[6, 16]]       # the smallest subnormal, both signs
    assert int(tiny[0]) == 1 and int(tiny[1]) == 0x8001
    want = 2.0 ** -24 if code == 2 else 2.0 ** -133
    assert RC.range_reference(tiny, code) == (0, int(np.array([want], dtype=np.float32).view(np.uint32)[0]))
