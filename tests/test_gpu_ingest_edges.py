"""GPU: the alignment ingest and the predictor-input packing, bit for bit, at every warp, tile and grid-stride edge
(tests/ingest_cases.py), through the C ABI wherever ingest_msa cannot reach a branch.

* rnamsm_msa_greedy_select: selected rows identical to oracle/msa_ingest_ref.greedy_select_indices in both modes.
* rnamsm_msa_clean after split_records: rows identical to the Bio.SeqIO restatement + clean_sequence; on a malformed
  file ``bad`` names a malformed record.
* rnamsm_msa_tokenize: tokens identical to a plain LUT gather (``encode`` for the vocabulary LUT), with and without
  a row list, all 256 byte values.
* rnamsm_ss_pack / rnamsm_rsa_pack: torch.equal to the restatements.

Outputs go into buffers poisoned with a sentinel (a NaN bit pattern no kernel makes), with guard regions on both
sides: the guards must come back untouched and nothing of the output may still hold the sentinel.  Every call runs
twice and must give the same bits.  Argument limits must fail before any launch, with a readable message.
"""
import functools
import os

import numpy as np
import pytest
import torch

import ingest_cases as IC
from oracle import msa_ingest_ref as I

pytestmark = pytest.mark.gpu

GUARD = 256
CASES = {c.name: c for c in IC.GREEDY_CASES}
FILES = IC.messy_files()


@pytest.fixture(scope="module")
def L():
    from rnamsm_b200 import _lib
    _lib.device_check(torch.device("cuda:0"))
    return _lib


def launches(L):
    torch.cuda.synchronize()
    return L.lib.rnamsm_launch_count()


class Guarded:
    """n elements between two GUARD-long regions, all filled with a sentinel word of the element's width."""

    def __init__(self, n, dtype, word):
        idt = {4: torch.int32, 8: torch.int64, 1: torch.uint8}[torch.empty(0, dtype=dtype).element_size()]
        self.bits = torch.full((GUARD + n + GUARD,), word, dtype=idt, device="cuda")
        self.out = self.bits.view(dtype)[GUARD:GUARD + n]
        self.word, self.n = word, n

    def check(self, what, written=True):
        g = torch.cat([self.bits[:GUARD], self.bits[GUARD + self.n:]])
        assert bool((g == self.word).all()), f"{what}: guard region written"
        if written:
            assert not bool((self.bits[GUARD:GUARD + self.n] == self.word).any()), f"{what}: element(s) never written"
        return self.out


NAN_WORD = 0x7FA5A5A5                  # a float32 NaN; kernel-made NaNs and every copied value have other bits


def twice(fn):
    """Run fn() twice; both results (tensors or tuples of tensors) must be the same bits."""
    a, b = fn(), fn()
    a, b = (a, b) if isinstance(a, tuple) else ((a,), (b,))
    for x, y in zip(a, b):
        assert torch.equal(x.view(torch.uint8) if x.dtype.is_floating_point else x,
                           y.view(torch.uint8) if y.dtype.is_floating_point else y), "second call differs"
    return a if len(a) > 1 else a[0]


# ------------------------------------------------------------------------------------------------ greedy select

@functools.lru_cache(maxsize=None)
def oracle_selection(name, mode):
    c = CASES[name]
    return I.greedy_select_indices(c.chars(), c.num, mode) if c.num < c.N else list(range(c.N))


def greedy(L, chars_d, num, want_max, poison):
    """The workspace starts as all `poison` bytes: a mismatch count never written reads as 0 or 65535."""
    N, Lc = chars_d.shape
    g = Guarded(num, torch.int32, -7)
    ws = torch.full((L.lib.rnamsm_msa_greedy_workspace(N, num),), poison, dtype=torch.uint8, device="cuda")
    L.check(L.lib.rnamsm_msa_greedy_select(L.ptr(chars_d), N, Lc, num, want_max, L.ptr(g.out), L.ptr(ws),
                                           L.stream_ptr()), "msa_greedy_select")
    torch.cuda.synchronize()
    return g.check("selected").clone()


@pytest.mark.parametrize("mode", ["max", "min"])
@pytest.mark.parametrize("name", list(CASES))
def test_greedy_select_matches_oracle(L, name, mode):
    c = CASES[name]
    chars = torch.from_numpy(c.chars()).cuda()
    n0 = launches(L)
    poisons = iter((0x00, 0xFF))
    sel = twice(lambda: greedy(L, chars, c.num, int(mode == "max"), next(poisons)))
    assert launches(L) - n0 == 2 * (3 * (c.num - 1) + 1)
    assert sel.cpu().tolist() == oracle_selection(name, mode), f"{name} {mode}"


def test_2drb_min_mode(L, msa_2drb_file):
    """BASELINE config 1's alignment through ingest_msa in "min" mode (the golden has the "max" selection only)."""
    import rnamsm_b200 as pkg
    chars = np.load(os.path.join(os.path.dirname(__file__), "golden", "ingest.npz"))["2drb_chars"]
    want = I.greedy_select_indices(chars, 512, "min")
    v = pkg.Vocab(pkg.Alphabet())
    tokens, rows = twice(lambda: pkg.ingest_msa(msa_2drb_file, v, max_seqs=512, sample_method="diversity-min"))
    assert rows.cpu().tolist() == want
    assert torch.equal(tokens.cpu(), torch.from_numpy(I.encode([bytes(chars[i]).decode() for i in want])))


# ------------------------------------------------------------------------------------------------ clean

def clean(L, raw, off, N, Lc, every_row):
    raw_d = torch.frombuffer(bytearray(raw + b"\0"), dtype=torch.uint8)[:len(raw)].cuda()
    off_d = torch.from_numpy(off).cuda()
    g = Guarded(N * Lc, torch.uint8, 0xA5)
    bad = torch.full((1,), -3, dtype=torch.int32, device="cuda")
    L.check(L.lib.rnamsm_msa_clean(L.ptr(raw_d), L.ptr(off_d), N, Lc, L.ptr(g.out), L.ptr(bad), L.stream_ptr()),
            "msa_clean")
    torch.cuda.synchronize()
    g.check("chars", written=every_row)
    return g.out.view(N, Lc).clone(), bad.clone()


@pytest.mark.parametrize("name", list(FILES))
def test_clean_matches_seqio(L, name, tmp_path):
    from rnamsm_b200.ingest import cleaned_length, split_records
    data, well_formed = FILES[name]
    p = tmp_path / "x.a2m"
    p.write_bytes(data)
    _, raw, off = split_records(str(p))
    rows = IC.reference_rows(data)
    N, Lc = len(rows), cleaned_length(raw[off[0]:off[1]])
    assert N == len(off) - 1 and Lc == len(rows[0])
    if Lc == 0:
        pytest.skip("first record cleans to nothing")
    chars, bad = twice(lambda: clean(L, raw, off, N, Lc, well_formed))
    chars = chars.cpu().numpy()
    good = [n for n, r in enumerate(rows) if len(r) == Lc]
    for n in good:
        assert bytes(chars[n]).decode("latin-1") == rows[n], f"{name}: record {n}"
    b = int(bad.item())
    if well_formed:
        assert b == 0 and len(good) == N
    else:
        assert b - 1 in set(range(N)) - set(good), f"{name}: bad names record {b - 1}, malformed: " \
                                                    f"{sorted(set(range(N)) - set(good))}"


@pytest.mark.parametrize("name", [n for n, (_, ok) in FILES.items() if ok])
def test_ingest_msa_reads_messy_files(name, tmp_path):
    import rnamsm_b200 as pkg
    p = tmp_path / "x.a2m"
    p.write_bytes(FILES[name][0])
    rows = IC.reference_rows(FILES[name][0])
    tokens, sel = pkg.ingest_msa(str(p), pkg.Vocab(pkg.Alphabet()), max_seqs=10 ** 6, max_seqlen=10 ** 6)
    assert sel.cpu().tolist() == list(range(len(rows)))
    assert torch.equal(tokens.cpu(), torch.from_numpy(I.encode(rows)))


# ------------------------------------------------------------------------------------------------ tokenize

def tokenize(L, chars_d, rows_d, R, lut_d, bos):
    Lc = chars_d.shape[1]
    g = Guarded(R * (Lc + 1), torch.int64, -5)
    L.check(L.lib.rnamsm_msa_tokenize(L.ptr(chars_d), Lc, L.ptr(rows_d), R, L.ptr(lut_d), bos, L.ptr(g.out),
                                      L.stream_ptr()), "msa_tokenize")
    torch.cuda.synchronize()
    return g.check("tokens").view(R, Lc + 1).clone()


@pytest.mark.parametrize("R,Lc,with_rows", IC.TOKENIZE_CASES)
def test_tokenize_matches_lut(L, R, Lc, with_rows):
    rng = np.random.default_rng(R * 1000 + Lc)
    n_src = R + 5 if with_rows else R
    chars = IC.all_bytes_chars(n_src, Lc, R + Lc)
    rows = rng.permutation(n_src)[:R].astype(np.int32) if with_rows else None
    chars_d = torch.from_numpy(chars).cuda()
    rows_d = torch.from_numpy(rows).cuda() if with_rows else None
    for lut, bos in ((IC.vocab_lut(), 0), (rng.permutation(256).astype(np.uint8), 201)):
        tok = twice(lambda: tokenize(L, chars_d, rows_d, R, torch.from_numpy(lut).cuda(), bos))
        assert torch.equal(tok.cpu(), torch.from_numpy(IC.tokenize_reference(chars, rows, lut, bos)))
        if bos == 0:
            sel = chars if rows is None else chars[rows]
            assert torch.equal(tok.cpu(), torch.from_numpy(I.encode([bytes(r).decode("latin-1") for r in sel])))


# ------------------------------------------------------------------------------------------------ packs

@pytest.mark.parametrize("Ls,start,K", IC.SS_CASES)
def test_ss_pack_matches_restatement(L, Ls, start, K):
    C = Ls + start
    rng = np.random.default_rng(Ls * 7 + K + start)
    maps = rng.random((K, C, C), dtype=np.float32)
    seq = IC.pack_sequence(Ls, Ls + K)
    want = torch.from_numpy(IC.ss_reference(maps[:, start:, start:], seq)).cuda()
    maps_d = torch.from_numpy(maps).cuda()
    codes = torch.from_numpy(IC.seq_codes(seq)).cuda()

    def run():
        g = Guarded((K + 8) * Ls * Ls, torch.float32, NAN_WORD)
        L.check(L.lib.rnamsm_ss_pack(L.ptr(maps_d), K, C, start, Ls, L.ptr(codes), L.ptr(g.out), L.stream_ptr()),
                "ss_pack")
        torch.cuda.synchronize()
        return g.check("ss_pack").view(1, K + 8, Ls, Ls).clone()

    assert torch.equal(twice(run), want)


@pytest.mark.parametrize("Ls,D,oh,extra", IC.RSA_CASES)
def test_rsa_pack_matches_oracle(L, Ls, D, oh, extra):
    import ctypes as C
    emb, mu, sd, mu_oh, sd_oh = IC.rsa_inputs(Ls, D, extra, Ls * 31 + D + extra)
    seq = IC.pack_sequence(Ls, D + Ls)
    want = torch.from_numpy(IC.rsa_reference(emb, D, seq, mu, sd, *((mu_oh, sd_oh) if oh else ()))).cuda()
    emb_d, mu_d, sd_d = (torch.from_numpy(a).cuda() for a in (emb, mu, sd))
    codes = torch.from_numpy(IC.seq_codes(seq)).cuda()
    oh_mu = (C.c_double * 4)(*mu_oh.tolist()) if oh else None
    oh_sd = (C.c_double * 4)(*sd_oh.tolist()) if oh else None
    n_ch = 4 * oh + D + 1

    def run():
        g = Guarded(n_ch * Ls, torch.float32, NAN_WORD)
        L.check(L.lib.rnamsm_rsa_pack(L.ptr(emb_d), D + extra, Ls, D, L.ptr(codes), oh_mu, oh_sd, L.ptr(mu_d),
                                      L.ptr(sd_d), L.ptr(g.out), L.stream_ptr()), "rsa_pack")
        torch.cuda.synchronize()
        return g.check("rsa_pack").view(1, n_ch, Ls).clone()

    assert torch.equal(twice(run), want)


def test_python_packs_take_lowercase_and_unknown_letters():
    """pack_ss_input / pack_rsa_input map every letter outside ACGU (lowercase included) to an all-zero one-hot."""
    import rnamsm_b200 as pkg
    seq = IC.pack_sequence(40, 3)
    rng = np.random.default_rng(4)
    Ls = len(seq)
    maps = rng.random((1, 2, 3, Ls + 1, Ls + 1), dtype=np.float32)
    x = pkg.pack_ss_input(torch.from_numpy(maps).cuda(), seq)
    want = IC.ss_reference(maps[0].reshape(6, Ls + 1, Ls + 1)[:, 1:, 1:], seq)
    assert torch.equal(x.cpu(), torch.from_numpy(want))
    emb, mu, sd, mu_oh, sd_oh = IC.rsa_inputs(Ls + 1, 64, 0, 5)
    rep = torch.from_numpy(emb).view(1, 1, Ls + 1, 64).cuda()
    x = pkg.pack_rsa_input(rep, seq, mu, sd, mu_oh, sd_oh)
    assert torch.equal(x.cpu(), torch.from_numpy(IC.rsa_reference(emb[1:], 64, seq, mu, sd, mu_oh, sd_oh)))


# ------------------------------------------------------------------------------------------------ argument limits

def test_argument_limits_fail_before_any_launch(L):
    chars = torch.zeros((8, 4), dtype=torch.uint8, device="cuda")
    sel = torch.empty(2048, dtype=torch.int32, device="cuda")
    ws = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    st = L.stream_ptr()
    n0 = launches(L)
    for N, Lc, num, what in ((2000, 4, 1025, b"num <= 1024"), (8, 4, 9, b"> depth"), (8, 25600, 2, b"too long"),
                             (8, 4, 0, b"num=0")):
        assert L.lib.rnamsm_msa_greedy_select(L.ptr(chars), N, Lc, num, 1, L.ptr(sel), L.ptr(ws), st) != 0
        assert what in L.lib.rnamsm_last_error(), L.lib.rnamsm_last_error()
    maps = torch.zeros(16, dtype=torch.float32, device="cuda")
    assert L.lib.rnamsm_ss_pack(L.ptr(maps), 1, 65536, 0, 65536, L.ptr(chars), L.ptr(maps), st) != 0
    assert b"ss_pack" in L.lib.rnamsm_last_error()
    assert L.lib.rnamsm_rsa_pack(L.ptr(maps), 3, 4, 4, None, None, None, L.ptr(maps), L.ptr(maps), L.ptr(maps), st) != 0
    assert b"ld=3" in L.lib.rnamsm_last_error()
    assert L.lib.rnamsm_msa_tokenize(L.ptr(chars), 4, None, 0, L.ptr(chars), 0, L.ptr(maps), st) != 0
    assert L.lib.rnamsm_msa_clean(L.ptr(chars), L.ptr(chars), 0, 4, L.ptr(chars), L.ptr(maps), st) != 0
    assert launches(L) == n0


def test_ingest_msa_refuses_more_than_1024_diverse_rows(tmp_path):
    import rnamsm_b200 as pkg
    p = tmp_path / "deep.a2m"
    p.write_bytes(IC.write_messy(IC._rows(1100, 12, 3), np.random.default_rng(0)))
    with pytest.raises(RuntimeError, match="num <= 1024"):
        pkg.ingest_msa(str(p), pkg.Vocab(pkg.Alphabet()), max_seqs=1025, sample_method="diversity-max")
