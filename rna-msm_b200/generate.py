"""Sequences generated from an alignment by iterative masked sampling with the LM head::

    python -m rnamsm_b200.generate --MSA_file X.a2m_msa2 --steps 200 --n_chains 4 --out gen.fasta \
        [--rows query|all] [--mask_prob 0.1] [--temperature 1.0] [--seed 0]

The alignment is read like ``rnamsm_b200.score`` reads it; its first row is the query.  Every chain starts from the
alignment and runs ``MSATransformer.sample_msa`` for ``--steps`` steps over the query row or over all rows.  Writes the
sampled rows of every chain as FASTA, with the BOS column and pads removed (a token without a one-letter form, such as
``<unk>``, as ``X``), under headers
``>chain<k>_row<r> source=<record index>``: chain ``k``, alignment row ``r``, and the index of that row's record in
``--MSA_file``.
"""
from __future__ import annotations

import argparse

from .ingest import ingest_msa
from .inference import build_model


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--MSA_file", required=True)
    ap.add_argument("--steps", type=int, required=True)
    ap.add_argument("--n_chains", type=int, default=1)
    ap.add_argument("--out", required=True, help="FASTA of the generated rows")
    ap.add_argument("--rows", default="query", choices=["query", "all"])
    ap.add_argument("--mask_prob", type=float, default=0.1)
    ap.add_argument("--temperature", type=float, default=1.0)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--device", default="cuda")
    ap.add_argument("--model_path", default=None, help="Lightning checkpoint ('state_dict'); random init if omitted")
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16", "bf16_pure", "tf32x3", "fp32"])
    ap.add_argument("--max_seqs_per_msa", type=int, default=512)
    ap.add_argument("--sample_method", default="first", choices=["first", "diversity-max", "diversity-min"])
    ap.add_argument("--max_seqlen", type=int, default=1024)
    ap.add_argument("--no_embed_positions_msa", action="store_true")
    a = ap.parse_args(argv)
    model, vocab = build_model(a.model_path, a.device, a.precision, embed_positions_msa=not a.no_embed_positions_msa,
                               max_seqlen=a.max_seqlen)
    tokens, sel = ingest_msa(a.MSA_file, vocab, a.max_seqs_per_msa, a.max_seqlen, a.sample_method, device=str(model.device))
    rows = [0] if a.rows == "query" else list(range(tokens.shape[0]))
    out = model.sample_msa(tokens, a.steps, mask_prob=a.mask_prob, temperature=a.temperature, rows=rows,
                           n_chains=a.n_chains, seed=a.seed).cpu()
    sel = sel.cpu().tolist()
    start = int(vocab.prepend_bos)
    letter = [t if len(t) == 1 else "X" for t in vocab.tokens]
    with open(a.out, "w") as f:
        for k in range(out.shape[0]):
            for r in rows:
                seq = "".join(letter[v] for v in out[k, r, start:].tolist() if v != vocab.pad_idx)
                f.write(f">chain{k}_row{r} source={sel[r]}\n{seq}\n")
    print(f"{out.shape[0]} chains x {len(rows)} rows, {a.steps} steps -> {a.out}")


if __name__ == "__main__":
    main()
