"""GPU: the sharded single-MSA forward (rna-msm_b200/sharded.py) through the C-ABI kernels.
world 1 (always): the per-phase ops must reproduce MSATransformer.forward exactly (same kernels, same
order).  world 2 (needs two GPUs; skipped otherwise): NCCL all-reduce of the tied logits + the two
all-to-all re-layouts against the single-GPU forward of the same model."""
import os
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import msa_ref as O  # noqa: E402

pytestmark = pytest.mark.gpu


def _model(pkg, layers, precision, device):
    vocab = pkg.Vocab(pkg.Alphabet())
    m = pkg.MSATransformer(vocab, num_layers=layers, precision=precision)
    m.load_state_dict(O.make_weights(9, num_layers=layers, sharpen=2.0), strict=True)
    return m.eval().to(device)


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
@pytest.mark.parametrize("pads", [(0, 0), (3, 2)], ids=["nopad", "pad"])
def test_world1_matches_model_forward(precision, pads):
    import rnamsm_b200 as pkg
    from rnamsm_b200.sharded import sharded_forward
    m = _model(pkg, 3, precision, "cuda")
    tokens = O.make_tokens(40, 70, 4, pad_cols=pads[0], pad_rows=pads[1]).cuda()
    ref = m(tokens, repr_layers=[3], need_head_weights=True, want_logits=False)
    out = sharded_forward(m, tokens)
    tol = 2e-6 if precision == "fp32" else 2e-3      # 16-bit: delta rounded once more to 16 bits on its way back
    assert O.rel_err(out["representations"][3].cpu(), ref["representations"][3].cpu()) < tol
    assert O.rel_err(out["row_attentions"].cpu(), ref["row_attentions"].cpu()) < tol


@pytest.mark.parametrize("pads", [(0, 0), (3, 2)], ids=["nopad", "pad"])
@pytest.mark.parametrize("scatter_fp32", ["0", "1"], ids=["delta16", "reduce32"])
def test_world1_fused_matches_model_forward(pads, scatter_fp32, monkeypatch):
    """The peer-memory kernels (softmax_p2p, layernorm_push, residual scatter in both payload modes,
    add_layernorm) with a single rank."""
    import rnamsm_b200 as pkg
    from rnamsm_b200 import sharded
    from rnamsm_b200.sharded import sharded_forward
    monkeypatch.setenv("RNAMSM_SCATTER_FP32", scatter_fp32)
    sharded._FUSED_CACHE.clear()
    m = _model(pkg, 3, "fp16", "cuda")
    tokens = O.make_tokens(40, 80, 4, pad_cols=pads[0], pad_rows=pads[1]).cuda()
    ref = m(tokens, repr_layers=[3], need_head_weights=True, want_logits=False)
    out = sharded_forward(m, tokens, fused=True)
    torch.cuda.synchronize()
    assert O.rel_err(out["representations"][3].cpu(), ref["representations"][3].cpu()) < 2e-3
    assert O.rel_err(out["row_attentions"].cpu(), ref["row_attentions"].cpu()) < 2e-3
    # results are fresh tensors: a second call (which rewrites the persistent peer buffers) must not change them
    keep_rep, keep_att = out["representations"][3].clone(), out["row_attentions"].clone()
    other = O.make_tokens(40, 80, 5).cuda()
    sharded_forward(m, other, fused=True)
    torch.cuda.synchronize()
    assert torch.equal(keep_rep, out["representations"][3]) and torch.equal(keep_att, out["row_attentions"])
    # host outputs: the owned map rows go to the shared host buffer in the *_atp.npy layout, emb to pinned memory
    from rnamsm_b200.sharded import ShardedHostOutput
    host = ShardedHostOutput(3, m.num_attention_heads, 80, m.embed_dim, start=1)
    out2 = sharded_forward(m, tokens, fused=True, host_out=host, gather_maps=False)
    assert out2["row_attentions_range"] == (0, 80)
    want = ref["row_attentions"][0, :, :, 1:, 1:].reshape(-1, 79, 79).cpu()
    assert O.rel_err(host.atp.clone(), want) < 2e-3
    assert O.rel_err(host.emb, ref["representations"][3][0, 0, 1:].cpu()) < 2e-3
    host.close()
    # a different shape reallocates the peer buffers; earlier results stay valid
    small = O.make_tokens(16, 32, 6).cuda()
    sharded_forward(m, small, fused=True)
    torch.cuda.synchronize()
    assert torch.equal(keep_rep, out["representations"][3])


@pytest.mark.parametrize("fused", [False, True], ids=["nccl", "fused"])
def test_world1_uneven_shape_is_padded_inside(fused):
    """Shapes the shard plan cannot split (here: C not a multiple of the fused schedule's 16-column boxes) are padded
    with <pad> inside the sharded forward and come back in the caller's shape, equal to the plain forward on every real
    token (align_scaling keeps the TRUE depth)."""
    import rnamsm_b200 as pkg
    from rnamsm_b200 import sharded
    from rnamsm_b200.sharded import ShardedHostOutput, pad_to_shards, sharded_forward
    sharded._FUSED_CACHE.clear()
    m = _model(pkg, 3, "fp16", "cuda")
    tokens = O.make_tokens(37, 71, 4).cuda()
    assert tuple(pad_to_shards(tokens, 1, 16, 1).shape) == (1, 37, 80) and pad_to_shards(tokens, 1, 1, 1) is tokens
    assert tuple(pad_to_shards(tokens, 8, 16, 1).shape) == (1, 40, 128)
    ref = m(tokens, repr_layers=[3], need_head_weights=True, want_logits=False)
    out = sharded_forward(m, tokens, fused=fused)
    torch.cuda.synchronize()
    assert tuple(out["representations"][3].shape) == (1, 37, 71, m.embed_dim) and out["row_shard"] == (0, 37)
    assert tuple(out["row_attentions"].shape[-2:]) == (71, 71)
    assert O.rel_err(out["representations"][3].cpu(), ref["representations"][3].cpu()) < 2e-3
    assert O.rel_err(out["row_attentions"].cpu(), ref["row_attentions"].cpu()) < 2e-3
    if fused:
        host = ShardedHostOutput(3, m.num_attention_heads, 71, m.embed_dim, start=1)
        out2 = sharded_forward(m, tokens, fused=True, host_out=host, gather_maps=False)
        assert out2["row_attentions_range"] == (0, 71) and tuple(out2["row_attentions_rows"].shape[-2:]) == (71, 71)
        want = ref["row_attentions"][0, :, :, 1:, 1:].reshape(-1, 70, 70).cpu()
        assert O.rel_err(host.atp.clone(), want) < 2e-3
        assert O.rel_err(host.emb, ref["representations"][3][0, 0, 1:].cpu()) < 2e-3
        host.close()


def _worker(rank, world, port, precision, q, shape=(64, 96)):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import rnamsm_b200 as pkg
        from rnamsm_b200.sharded import sharded_forward
        m = _model(pkg, 3, precision, f"cuda:{rank}")
        tokens = O.make_tokens(shape[0], shape[1], 4, pad_cols=2, pad_rows=2).to(f"cuda:{rank}")
        ref = m(tokens, repr_layers=[3], need_head_weights=True, want_logits=False)
        if shape[0] % world or shape[1] % (16 * world):
            # padded inside: what is computed AT <pad> positions differs (and is read by nobody); compare the real tokens
            keep = tokens.ne(m.vocab.pad_idx).unsqueeze(-1).float()
            ref["representations"][3] = ref["representations"][3] * keep
        else:
            keep = None
        mask = (lambda rep, r0=0, r1=None: rep if keep is None else rep * keep[:, r0:r1])
        out = sharded_forward(m, tokens, gather_rows=True)
        torch.cuda.synchronize()
        errs = [O.rel_err(mask(out["representations"][3]).cpu(), ref["representations"][3].cpu()),
                O.rel_err(out["row_attentions"].cpu(), ref["row_attentions"].cpu())]
        if precision == "fp16":                    # fused peer-memory schedule: row shard + full maps on every rank
            fo = sharded_forward(m, tokens, fused=True)
            torch.cuda.synchronize()
            r0, r1 = fo["row_shard"]
            errs.append(O.rel_err(mask(fo["representations"][3], r0, r1).cpu(), ref["representations"][3][:, r0:r1].cpu()))
            errs.append(O.rel_err(fo["row_attentions"].cpu(), ref["row_attentions"].cpu()))
            # host outputs: every rank DMAs the map rows it owns into the shared host buffer; emb on rank 0
            from rnamsm_b200.sharded import ShardedHostOutput
            host = ShardedHostOutput(3, m.num_attention_heads, tokens.shape[-1], m.embed_dim, start=1, group=None)
            for _ in range(2):                     # twice: the second call reuses the peer buffers and the flag epochs
                fo2 = sharded_forward(m, tokens, fused=True, host_out=host, gather_maps=False)
            i0, i1 = fo2["row_attentions_range"]
            assert fo2["row_attentions_rows"].shape[2] == i1 - i0
            L_ = tokens.shape[-1] - 1
            want_atp = ref["row_attentions"][0, :, :, 1:, 1:].reshape(-1, L_, L_).cpu()
            errs.append(O.rel_err(mask(fo2["representations"][3], r0, r1).cpu(), ref["representations"][3][:, r0:r1].cpu()))
            errs.append(O.rel_err(host.atp.clone(), want_atp))       # complete on EVERY rank (shared memory)
            if rank == 0:
                emb = host.emb if keep is None else host.emb * keep[0, 0, 1:].cpu()
                errs.append(O.rel_err(emb, ref["representations"][3][0, 0, 1:].cpu()))
                errs.append(0.0)
            host.close()
        q.put((rank, max(errs[0::2]), max(errs[1::2])))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("shape", [(64, 96), (63, 91)], ids=["even", "uneven"])
@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_world2_nccl_matches_single_gpu(precision, shape):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29710 + (os.getpid() % 200)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, precision, q, shape)) for r in range(2)]
    for p in procs:
        p.start()
    results = [q.get(timeout=300) for _ in range(2)]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    tol = 2e-5 if precision == "fp32" else 3e-3
    for rank, e_rep, e_att in results:
        assert e_rep < tol and e_att < tol, (rank, e_rep, e_att)
