"""GPU: full-length features from overlapping windows (``MSATransformer.forward_windows``,
``rnamsm_msa_forward_windows``, ``extract_features_windowed``, ``run_inference(long_mode="window")``).

Most tests use a model whose learned positions stop at 64 (``max_seqlen=64``, ``embed_positions.weight`` cut from the
oracle's weights), so windows engage at L of about 100 to 200.  Every window's outputs come from ``forward`` of its
grid: entries one window holds are bit-identical to it, every entry follows the float64 restatement of the stitching
(windows_ref.py) applied to those forwards, and pairs no window holds are exactly 0."""
import numpy as np
import pytest
import torch

from oracle import msa_ref as O
import windows_ref as WR

pytestmark = pytest.mark.gpu

SMALL_SEQLEN = 64            # learned positions of the small model: windows of at most 63 residues
LAYERS = 2
STITCH_TOL = 1e-5            # fp32 accumulation against float64, relative to the largest value of the output


@pytest.fixture(scope="module")
def pkg():
    import rnamsm_b200
    return rnamsm_b200


def build_small(pkg, seed, precision, layers=LAYERS, max_seqlen=SMALL_SEQLEN):
    model = pkg.MSATransformer(pkg.Vocab(pkg.Alphabet()), num_layers=layers, max_seqlen=max_seqlen, precision=precision)
    sd = O.make_weights(int(seed), num_layers=layers, sharpen=2.0)
    sd["embed_positions.weight"] = sd["embed_positions.weight"][:max_seqlen + O.PAD_IDX + 1].clone()
    model.load_state_dict(sd, strict=True)
    return model.eval().cuda()


def window_forwards(model, t, starts, W, contacts=True):
    """-> (embs [K, W, D], maps [K, NH, W, W], contacts [K, W, W]) float32 numpy, from forward of each window grid."""
    N = model.num_layers
    embs, maps, cons = [], [], []
    for s in starts:
        g = torch.cat([t[:, :1], t[:, 1 + s:1 + s + W]], dim=1)
        r = model(g.unsqueeze(0), repr_layers=[N], need_head_weights=True, return_contacts=contacts, want_logits=False)
        emb, atp = model_features(r, model)
        embs.append(emb)
        maps.append(atp)
        if contacts:
            cons.append(r["contacts"][0].cpu().numpy())
    return np.stack(embs), np.stack(maps), (np.stack(cons) if contacts else None)


def model_features(r, model):
    from rnamsm_b200 import extract_features
    return extract_features(r, model.vocab, model.num_layers)


def check_against_windows(out, embs, maps, cons, starts, L):
    W = embs.shape[1]
    emb, atp = out["emb"].cpu().numpy(), out["atp"].cpu().numpy()
    con = out["contacts"].cpu().numpy() if cons is not None else None
    assert emb.shape == (L, embs.shape[2]) and atp.shape == (maps.shape[1], L, L)
    # entries one window holds: that window's value bit for bit
    n_res = np.zeros(L, dtype=np.int64)
    for s in starts:
        n_res[s:s + W] += 1
    one = WR.single(L, W, starts)
    for k, s in enumerate(starts):
        rows = np.nonzero(n_res[s:s + W] == 1)[0]
        assert np.array_equal(emb[s + rows], embs[k][rows]), k
        m = one[s:s + W, s:s + W] == k
        assert np.array_equal(atp[:, s:s + W, s:s + W][:, m], maps[k][:, m]), k
        if con is not None:
            assert np.array_equal(con[s:s + W, s:s + W][m], cons[k][m]), k
    # every entry: the float64 restatement
    ref_emb, ref_atp, ref_con = WR.stitch(embs, maps, starts, L, cons)
    for got, ref in ((emb, ref_emb), (atp, ref_atp), (con, ref_con)):
        if got is None:
            continue
        err = np.abs(got - ref).max() / max(np.abs(ref).max(), 1e-30)
        assert err <= STITCH_TOL, err
    # pairs no window holds: exactly 0
    cov = WR.covered(L, W, starts)
    assert not atp[:, ~cov].any()
    if con is not None:
        assert not con[~cov].any()


# ------------------------------------------------------------------------------------------------ windows vs forward
CASES = {
    "R6_L150_w63_s31": dict(R=6, L=150, window=63, stride=31),
    "R6_L150_w63_s63_pad": dict(R=6, L=150, window=63, stride=63, pad_cols=3),
    "R4_L100_w48_s1": dict(R=4, L=100, window=48, stride=1),
    "R5_L120_w40_s13_pad_rows": dict(R=5, L=120, window=40, stride=13, pad_cols=2, pad_rows=1),
    "R1_L130_w63_s31": dict(R=1, L=130, window=63, stride=31),
}


def case_tokens(c, seed):
    return O.make_tokens(c["R"], c["L"] + 1, seed, pad_cols=c.get("pad_cols", 0), pad_rows=c.get("pad_rows", 0),
                         gap_p=0.1)[0]


@pytest.mark.parametrize("name", list(CASES))
@pytest.mark.parametrize("precision", ["fp16", "bf16", "fp32", "tf32x3"])
def test_windows_match_forward_of_each_window(pkg, name, precision):
    c = CASES[name]
    model = build_small(pkg, 7, precision)
    t = case_tokens(c, 3).cuda()
    L, window, stride = c["L"], c["window"], c["stride"]
    out = model.forward_windows(t, window=window, stride=stride, return_contacts=True)
    starts = WR.window_starts(L, window, stride)
    assert out["window_starts"] == starts
    for k in ("emb", "atp", "contacts"):
        assert out[k].dtype == torch.float32 and out[k].is_cuda
    embs, maps, cons = window_forwards(model, t, starts, min(window, L))
    check_against_windows(out, embs, maps, cons, starts, L)


# ------------------------------------------------------------------------------------------------ short inputs
@pytest.mark.parametrize("precision", ["fp16", "bf16", "fp32", "tf32x3"])
@pytest.mark.parametrize("R,L,pad_cols,window", [(6, 50, 0, None), (5, 63, 2, None), (1, 40, 0, 48), (6, 30, 0, 30)])
def test_short_input_equals_forward(pkg, precision, R, L, pad_cols, window):
    model = build_small(pkg, 5, precision)
    t = O.make_tokens(R, L + 1, 2, pad_cols=pad_cols, gap_p=0.1)[0].cuda()
    out = model.forward_windows(t, window=window, return_contacts=True)
    r = model(t.unsqueeze(0), repr_layers=[model.num_layers], need_head_weights=True, return_contacts=True,
              want_logits=False)
    emb, atp = model_features(r, model)
    assert out["window_starts"] == [0]
    assert np.array_equal(out["emb"].cpu().numpy(), emb)
    assert np.array_equal(out["atp"].cpu().numpy(), atp)
    assert torch.equal(out["contacts"], r["contacts"][0])
    e2, a2 = pkg.extract_features_windowed(model, t.unsqueeze(0), window=window)
    assert np.array_equal(e2, emb) and np.array_equal(a2, atp)


# ------------------------------------------------------------------------------------------------ grouping
@pytest.mark.parametrize("precision,R", [("fp16", 6), ("bf16", 3), ("fp32", 4), ("fp16", 1)])
def test_grouping_does_not_change_the_bits(pkg, precision, R):
    model = build_small(pkg, 9, precision)
    L, window, stride = 170, 63, 25
    t = O.make_tokens(R, L + 1, 4, pad_cols=1, gap_p=0.1)[0].cuda()
    K = len(WR.window_starts(L, window, stride))
    T = R * (window + 1)
    outs = [model.forward_windows(t, window=window, stride=stride, return_contacts=True, token_budget=g * T)
            for g in (1, 2, 3, K)]
    for o in outs[1:]:
        for k in ("emb", "atp", "contacts"):
            assert torch.equal(o[k], outs[0][k]), k


# ------------------------------------------------------------------------------------------------ full-size model
def test_full_size_model_default_window(pkg):
    """The shipped shape: 10 layers, 1023 learned positions, 32 x 1501, default window 1023 and stride 511."""
    sd = O.make_weights(42, sharpen=2.0)
    model = pkg.MSATransformer(pkg.Vocab(pkg.Alphabet()), num_layers=10, precision="fp16")
    model.load_state_dict(sd, strict=True)
    model = model.eval().cuda()
    L = 1501
    t = O.make_tokens(32, L + 1, 6, gap_p=0.1)[0].cuda()
    with pytest.raises(IndexError):
        model(t.unsqueeze(0), want_logits=False)
    out = model.forward_windows(t)
    starts = out["window_starts"]
    assert starts == [0, 478]
    assert out["emb"].shape == (L, 768) and out["atp"].shape == (120, L, L)
    embs, maps, _ = window_forwards(model, t, starts, 1023, contacts=False)
    heads = [0, 57, 119]                                     # the float64 restatement on a few maps keeps the host quick
    sub = {"emb": out["emb"], "atp": out["atp"][heads]}
    check_against_windows(sub, embs, maps[:, heads], None, starts, L)
    one = WR.single(L, 1023, starts)
    atp = out["atp"]
    for k, s in enumerate(starts):                           # every map, where one window holds the pair
        m = torch.from_numpy(one[s:s + 1023, s:s + 1023] == k).cuda()
        got = atp[:, s:s + 1023, s:s + 1023][:, m]
        assert torch.equal(got, torch.from_numpy(maps[k]).cuda()[:, m]), k


# ------------------------------------------------------------------------------------------------ end to end
def write_a2m(path, n, L, seed):
    rng = np.random.default_rng(seed)
    seqs = ["".join(rng.choice(list("ACGU-"), size=L, p=[0.24, 0.24, 0.24, 0.24, 0.04])) for _ in range(n)]
    with open(path, "w") as f:
        for i, s in enumerate(seqs):
            f.write(f">seq{i}\n{s}\n")
    return seqs[0]


def test_run_inference_long_window_and_crop(pkg, tmp_path):
    from rnamsm_b200 import inference
    L, D = 1100, 768
    d = tmp_path / "results"
    d.mkdir()
    seq = write_a2m(d / "long1.a2m_msa2", 8, L, 0)
    (tmp_path / "ids.txt").write_text("long1\n")
    base = ["--root_path", str(tmp_path), "--MSA_path", "results", "--MSA_list", "ids.txt", "--max_seqs_per_msa", "8"]
    inference.main(base + ["--long", "window"])
    emb, atp = np.load(d / "long1_emb.npy"), np.load(d / "long1_atp.npy")
    assert emb.shape == (L, D) and atp.shape == (120, L, L) and emb.dtype == atp.dtype == np.float32
    assert np.isfinite(emb).all() and np.isfinite(atp).all()
    cov = WR.covered(L, 1023, WR.window_starts(L, 1023, 511))
    assert not atp[:, ~cov].any() and (atp[:, cov] > 0).all()
    # the stitched outputs feed the downstream packers unchanged
    atp_d, emb_d = torch.from_numpy(atp).cuda(), torch.from_numpy(emb).cuda()
    ss = pkg.pack_ss_input(atp_d.view(1, 10, 12, L, L), seq.replace("-", "X"), prepend_bos=False)
    assert ss.shape == (1, 128, L, L) and torch.equal(ss[0, 8:], atp_d)
    rng = np.random.default_rng(1)
    mu, sd = rng.standard_normal(D).astype(np.float32), (1 + rng.random(D)).astype(np.float32)
    rsa = pkg.pack_rsa_input(emb_d.view(1, 1, L, D), seq.replace("-", "X"), mu, sd, prepend_bos=False)
    assert rsa.shape == (1, D + 1, L) and torch.isfinite(rsa).all()
    # crop: what the reference writes, the first 1023 columns
    inference.main(base)
    emb_c, atp_c = np.load(d / "long1_emb.npy"), np.load(d / "long1_atp.npy")
    assert emb_c.shape == (1023, D) and atp_c.shape == (120, 1023, 1023)
    model, vocab = inference.build_model(None)
    tokens, _ = pkg.ingest_msa(str(d / "long1.a2m_msa2"), vocab, 8, 1024, device=str(model.device))
    e_ref, a_ref = pkg.extract_features(model(tokens.unsqueeze(0), repr_layers=[10], need_head_weights=True,
                                              want_logits=False), vocab, 10)
    assert np.array_equal(emb_c, e_ref) and np.array_equal(atp_c, a_ref)


# ------------------------------------------------------------------------------------------------ errors
def test_argument_errors(pkg):
    model = build_small(pkg, 1, "fp16")
    t = O.make_tokens(4, 101, 1)[0].cuda()
    for kw, match in ((dict(window=64), "stride <= window"), (dict(window=10, stride=11), "stride <= window"),
                      (dict(window=10, stride=0), "stride <= window"), (dict(window=0), "stride <= window"),
                      (dict(token_budget=0), "token_budget")):
        with pytest.raises(ValueError, match=match):
            model.forward_windows(t, **kw)
    with pytest.raises(ValueError, match="one MSA"):
        model.forward_windows(torch.stack([t, t]))
    with pytest.raises(ValueError, match="no residues"):
        model.forward_windows(t[:, :1])
    with pytest.raises(RuntimeError, match="CUDA"):
        model.forward_windows(t.cpu())
    eos = build_small(pkg, 1, "fp16")
    eos.vocab = pkg.Vocab(pkg.Alphabet(append_eos=True))
    with pytest.raises(ValueError, match="EOS"):
        eos.forward_windows(t)


def test_too_large_fails_before_any_launch(pkg):
    model = build_small(pkg, 1, "fp16")
    t = O.make_tokens(2, 100_001, 1)[0].cuda()              # 24 maps of 10^10 entries: 960 GB
    model.forward_windows(t[:, :200])                       # warm: weights staged, modules loaded
    torch.cuda.synchronize()
    c0 = pkg._lib.lib.rnamsm_launch_count()
    with pytest.raises(torch.OutOfMemoryError):
        model.forward_windows(t)
    assert pkg._lib.lib.rnamsm_launch_count() == c0


# ------------------------------------------------------------------------------------------------ launches
def launches(pkg):
    return pkg._lib.lib.rnamsm_launch_count()


@pytest.mark.parametrize("precision,R", [("fp16", 6), ("fp32", 6), ("fp16", 1)])
@pytest.mark.parametrize("contacts", [False, True])
def test_launch_counts(pkg, precision, R, contacts):
    """Per pass: one window build and one stitch (read with rnamsm_profile_collect), the layer route of its grids
    (rnamsm_msa_forward_batch of the pass's grids, or one forward per grid, without the final LayerNorm), a row gather
    when R >= 2, one final LayerNorm, and the contact head's three launches per window when contacts are wanted."""
    L_ = pkg._lib
    model = build_small(pkg, 2, precision)
    L, window, stride = 150, 63, 31                          # four windows, two passes of two
    t = O.make_tokens(R, L + 1, 8)[0].cuda()
    budget = 2 * R * (window + 1)
    run = lambda: model.forward_windows(t, window=window, stride=stride, return_contacts=contacts, token_budget=budget)
    run()                                                    # warm
    g = t[:, :window + 1]
    batch = precision != "fp32" and R >= 2
    torch.cuda.synchronize()
    c0 = launches(pkg)
    if batch:
        model.forward_batch([g, g])
    else:
        model(g.unsqueeze(0), want_logits=False)
    c1 = launches(pkg)
    L_.profile_enable(True)
    run()
    c2 = launches(pkg)
    torch.cuda.synchronize()
    prof = L_.profile_collect()
    L_.profile_enable(False)
    assert prof["window_build"][1] == 2 and prof["window_stitch"][1] == 2
    route = 2 * (c1 - c0 - 1) if batch else 4 * (c1 - c0 - 1)
    assert c2 - c1 == route + 2 * (1 + (R >= 2) + 1 + 1) + (3 * 4 if contacts else 0)
