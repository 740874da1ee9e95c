"""CPU: host-side logic of the drop-in boundary -- state-dict schema, constructor surface,
tokenisation, error behaviour without a GPU (no fallback), output post-processing."""
import os

import numpy as np
import pytest
import torch

from oracle import msa_ref as O


@pytest.fixture(scope="module")
def pkg():
    import rnamsm_b200
    return rnamsm_b200


def test_state_dict_schema_matches_reference(pkg):
    vocab = pkg.Vocab(pkg.Alphabet())
    model = pkg.MSATransformer(vocab, num_layers=10)
    sd = model.state_dict()
    spec = O.state_dict_spec()
    assert len(sd) == 275 == len(spec)
    assert list(sd.keys()) == [n for n, _, _ in spec] or set(sd.keys()) == {n for n, _, _ in spec}
    for name, shape, _ in spec:
        assert tuple(sd[name].shape) == shape, name
    assert sum(p.numel() for p in model.parameters()) == 95_911_301
    assert model.msa_position_embedding.shape == (1, 1024, 1, 1)      # scalar per row (model.py:293-296)
    assert model.lm_head.weight is model.embed_tokens.weight           # tied
    missing = model.load_state_dict(O.make_weights(0), strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    m2 = pkg.MSATransformer(vocab, num_layers=1, embed_positions_msa=False)
    assert m2.msa_position_embedding is None and "msa_position_embedding" not in m2.state_dict()


def test_alphabet_and_tokenisation(pkg):
    a = pkg.Alphabet.from_architecture("rna language")
    assert a.all_toks == list(O.ALL_TOKS)
    v = pkg.Vocab.from_esm_alphabet(a)
    assert (len(v), v.pad_idx, v.eos_idx, v.prepend_bos, v.append_eos) == (12, 1, 2, True, False)
    tok = v.encode(["AGCU-XN", "agT.Z*-"])
    assert tok.dtype == np.int64 and tok.shape == (2, 8)
    assert tok[0].tolist() == [0, 4, 5, 6, 7, 10, 8, 9]
    assert tok[1].tolist() == [0, 3, 3, 3, 3, 3, 3, 10]   # raw encode: unknown symbols -> <unk>
    with pytest.raises(ValueError):
        v.encode(["AG", "A"])
    with pytest.raises(ValueError):
        pkg.Alphabet.from_architecture("ESM-1b")


def test_read_msa_cleaning_rules(pkg, tmp_path):
    p = tmp_path / "x.a2m_msa2"
    p.write_text(">q\nAGCTagc.N\n>h1 desc\nRY-U*AGC\nA\n")
    names, seqs = pkg.read_msa(str(p))
    assert names == ["q", "h1 desc"]
    assert seqs == ["AGCUX", "XX-UAGCA"]
    _, otok = O.read_a2m(str(tmp_path / "x.a2m_msa2"), 1)
    v = pkg.Vocab(pkg.Alphabet())
    assert np.array_equal(v.encode(seqs[:1]), otok.numpy())


def test_tokenize_matches_golden_2drb(pkg, golden_dir, msa_2drb_file):
    v = pkg.Vocab(pkg.Alphabet())
    tok = pkg.tokenize_msa(msa_2drb_file, v, 512, 1024)
    g = np.load(os.path.join(golden_dir, "2DRB_1.npz"))
    assert np.array_equal(tok.numpy(), g["tokens"][0].astype(np.int64))


def test_no_cpu_fallback(pkg):
    vocab = pkg.Vocab(pkg.Alphabet())
    model = pkg.MSATransformer(vocab, num_layers=1).eval()
    tokens = O.make_tokens(3, 5, 0)
    with pytest.raises(RuntimeError, match="CUDA"):
        model(tokens)
    layer = pkg.AxialTransformerLayer(768, 3072, 12).eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        layer(torch.zeros(2, 3, 1, 768))
    with pytest.raises(RuntimeError, match="CUDA"):
        layer.feed_forward_layer.layer(torch.zeros(2, 3, 1, 768))
    with pytest.raises(RuntimeError, match="CUDA"):
        model.forward_batch([tokens, tokens])
    with pytest.raises(ValueError):
        pkg.RowSelfAttention(768, 8)          # head_dim must be 64
    with pytest.raises(ValueError):
        model.set_precision("int8")
    assert model.set_precision("fp16").precision == "fp16"
    model.set_precision("bf16")


def test_extract_features_format(pkg):
    """RNA_MSM_Inference.py:150-166 layout: atp (120, L, L) f32 with index layer*12+head; emb (L, 768)."""
    v = pkg.Vocab(pkg.Alphabet())
    Cc, N, Hh = 7, 10, 12
    ra = torch.arange(N * Hh, dtype=torch.float32).view(1, N, Hh, 1, 1).expand(1, N, Hh, Cc, Cc).contiguous()
    rep = torch.randn(1, 4, Cc, 768)
    emb, atp = pkg.extract_features({"row_attentions": ra, "representations": {N: rep}}, v, N)
    assert atp.shape == (120, 6, 6) and atp.dtype == np.float32
    assert np.array_equal(atp[:, 0, 0], np.arange(120, dtype=np.float32))
    assert emb.shape == (6, 768) and np.array_equal(emb, rep[0, 0, 1:].numpy())
    o_emb, o_atp = O.extract_features({"row_attentions": ra, "representations": {N: rep}}, N)
    assert np.array_equal(o_emb, emb) and np.array_equal(o_atp, atp)


def test_shipped_fixture_format(pkg, golden_dir):
    """Format pin against the reference's shipped outputs results/2DRB_1_{atp,emb}.npy (values need the unpublished
    checkpoint): their shapes are stored in tests/golden/2DRB_1.npz, and extract_features on forward outputs shaped
    for the 512 x 36 token grid must produce arrays of those shapes in float32."""
    g = np.load(os.path.join(golden_dir, "2DRB_1.npz"))
    atp_shape, emb_shape = tuple(g["shipped_atp_shape"]), tuple(g["shipped_emb_shape"])
    assert atp_shape == (120, 35, 35) and emb_shape == (35, 768)
    assert g["atp"].dtype == g["emb"].dtype == np.float32
    R, Cc = g["tokens"].shape[1:]
    out = {"row_attentions": torch.rand(1, 10, 12, Cc, Cc), "representations": {10: torch.randn(1, R, Cc, 768)}}
    emb, atp = pkg.extract_features(out, pkg.Vocab(pkg.Alphabet()), 10)
    assert atp.shape == atp_shape and atp.dtype == np.float32
    assert emb.shape == emb_shape and emb.dtype == np.float32


def test_plan_batches_covers_every_msa_once_within_budget():
    """Grouping policy of extract_features_batch (8f row 4): every MSA exactly once, groups within the token
    budget unless a single alignment exceeds it, largest alignment first."""
    import random
    from rnamsm_b200.inference import plan_batches
    rnd = random.Random(3)
    shapes = [(256, rnd.randint(51, 501)) for _ in range(64)] + [(512, 600)]
    groups = plan_batches(shapes, 262144)
    assert sorted(i for g in groups for i in g) == list(range(len(shapes)))
    for g in groups:
        tok = sum(shapes[i][0] * shapes[i][1] for i in g)
        assert tok <= 262144 or len(g) == 1
    assert groups[0] == [64]                                               # 307200 tokens: alone, first
    assert len(groups) < len(shapes) // 2                                  # short alignments do get grouped
    assert plan_batches([], 10) == []


def test_plan_batches_properties():
    """hypothesis: any list of shapes and any budget -> a partition of the indices; no group over budget unless it
    is a single alignment; groups ordered by their largest member (largest first)."""
    from hypothesis import given, settings, strategies as st
    from rnamsm_b200.inference import plan_batches

    @settings(max_examples=200, deadline=None)
    @given(st.lists(st.tuples(st.integers(1, 1024), st.integers(1, 1024)), max_size=40), st.integers(1, 1 << 20))
    def check(shapes, budget):
        groups = plan_batches(shapes, budget)
        assert sorted(i for g in groups for i in g) == list(range(len(shapes)))
        tok = lambda i: shapes[i][0] * shapes[i][1]
        for g in groups:
            assert len(g) == 1 or sum(tok(i) for i in g) <= budget
            assert tok(g[0]) == max(tok(i) for i in g)
        heads = [tok(g[0]) for g in groups]
        assert heads == sorted(heads, reverse=True)

    check()


def test_shard_plan_properties():
    """hypothesis: the row / column ranges of the ranks tile the grid exactly, and the traffic model is symmetric."""
    from hypothesis import given, settings, strategies as st
    from rnamsm_b200.sharded import ShardPlan

    @settings(max_examples=100, deadline=None)
    @given(st.integers(1, 8), st.integers(1, 64), st.integers(1, 64))
    def check(n, a, b):
        R, C = a * n, b * n
        plans = [ShardPlan(R, C, n, r) for r in range(n)]
        rows = [i for p in plans for i in range(R)[p.rows()]]
        cols = [i for p in plans for i in range(C)[p.cols()]]
        assert rows == list(range(R)) and cols == list(range(C))
        assert all(p.rows(g) == plans[g].rows() and p.cols(g) == plans[g].cols() for p in plans for g in range(n))
        by = plans[0].bytes_per_layer()
        assert by["all_to_all_fwd"] == by["all_to_all_back"] == (R // n) * C * 768 * 2 * (n - 1) // n
        assert (by["logit_all_reduce"] == 0) == (n == 1)

    check()
