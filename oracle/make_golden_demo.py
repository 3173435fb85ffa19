"""Fixtures for the notebook-level boundary (TEST INFRASTRUCTURE; build container only: needs /root/reference).

Writes, from the UNMODIFIED reference tree:
  tests/golden/textcleaner_vocab.json   the 178-entry symbol table of text_utils.py and the ids of three val_list rows
  tests/golden/notebook_cells.json      the SOURCE of the inference cells of the two Demo notebooks, verbatim, so that
                                        tests/test_gpu_demo.py can exec() them over this package's modules
  tests/golden/plbert_real_slice.npz    a channel slice of the bundled PL-BERT checkpoint (Utils/PLBERT/step_1000000.t7,
                                        loads under torch.load(weights_only=True)) rounded to fp16: two of its twelve
                                        attention heads, 128 of the 768 hidden channels, 128 of the 2048 FFN channels, 64 of
                                        the 128 embedding channels and the first 96 positions, chosen so that the extreme
                                        values of the checkpoint (key bias up to 13, LayerNorm gains ~3) stay in.  The
                                        full checkpoint is 12 MB even in fp16; the slice is a 12-layer ALBERT of the same
                                        structure with the real value distribution in ~0.3 MB.  With it: token rows from
                                        Data/val_list.txt (cut to 96 tokens) and a seeded sample of transformers.AlbertModel's
                                        last_hidden_state rows on them WITH THE SAME fp16-rounded weights
"""
import json
import os
import sys

import numpy as np
import torch
import yaml

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
REF = os.environ.get("STYLETTS2_REFERENCE", "/root/reference")
GOLD = os.path.join(ROOT, "tests", "golden")

# the slice of the checkpoint that is stored (module docstring)
SLICE = dict(hidden_size=128, num_attention_heads=2, intermediate_size=128, embedding_size=64, max_position_embeddings=96)
SLICE_ROWS = 64   # sampled rows of last_hidden_state stored as the expected output


def _pick(n, k, score, n_top, g):
    """k of n indices, sorted: the n_top with the largest score, the rest a seeded draw from the others."""
    top = torch.argsort(score, descending=True)[:n_top]
    rest = torch.tensor([i for i in range(n) if i not in set(top.tolist())])
    rest = rest[torch.randperm(len(rest), generator=g)[:k - n_top]]
    return torch.sort(torch.cat([top, rest])).values


def slice_plbert(sd, seed=0):
    """Channel slice of an ALBERT state dict (keys as PLBert / AlbertModel) to the SLICE sizes."""
    g = torch.Generator().manual_seed(seed)
    p = "encoder.albert_layer_groups.0.albert_layers.0."
    a = lambda n: sd[p + n].float().abs()   # noqa: E731
    hd = 64
    # two whole heads: the one holding the largest |key bias| and the next one by that measure
    head_score = a("attention.key.bias").view(-1, hd).amax(1)
    heads = torch.argsort(head_score, descending=True)[:SLICE["num_attention_heads"]].sort().values
    i_att = torch.cat([torch.arange(h * hd, (h + 1) * hd) for h in heads.tolist()])
    # hidden channels: the most extreme gains / biases on the residual stream, then a seeded draw
    h_score = torch.stack([a("full_layer_layer_norm.weight"), a("full_layer_layer_norm.bias"), a("attention.LayerNorm.weight"),
                           a("attention.LayerNorm.bias"), a("attention.dense.bias"), a("ffn_output.bias")]).amax(0)
    i_h = _pick(sd[p + "full_layer_layer_norm.weight"].numel(), SLICE["hidden_size"], h_score, 32, g)
    i_f = _pick(sd[p + "ffn.bias"].numel(), SLICE["intermediate_size"], a("ffn_output.weight").amax(0), 16, g)
    e_score = sd["embeddings.LayerNorm.weight"].float().abs()
    i_e = _pick(e_score.numel(), SLICE["embedding_size"], e_score, 8, g)
    P = SLICE["max_position_embeddings"]
    rows_cols = {
        "embeddings.word_embeddings.weight": (None, i_e), "embeddings.position_embeddings.weight": (torch.arange(P), i_e),
        "embeddings.token_type_embeddings.weight": (None, i_e), "embeddings.LayerNorm.weight": (i_e,), "embeddings.LayerNorm.bias": (i_e,),
        "encoder.embedding_hidden_mapping_in.weight": (i_h, i_e), "encoder.embedding_hidden_mapping_in.bias": (i_h,),
        p + "full_layer_layer_norm.weight": (i_h,), p + "full_layer_layer_norm.bias": (i_h,),
        p + "attention.query.weight": (i_att, i_h), p + "attention.query.bias": (i_att,),
        p + "attention.key.weight": (i_att, i_h), p + "attention.key.bias": (i_att,),
        p + "attention.value.weight": (i_att, i_h), p + "attention.value.bias": (i_att,),
        p + "attention.dense.weight": (i_h, i_att), p + "attention.dense.bias": (i_h,),
        p + "attention.LayerNorm.weight": (i_h,), p + "attention.LayerNorm.bias": (i_h,),
        p + "ffn.weight": (i_f, i_h), p + "ffn.bias": (i_f,), p + "ffn_output.weight": (i_h, i_f), p + "ffn_output.bias": (i_h,),
        "pooler.weight": (i_h, i_h), "pooler.bias": (i_h,),
    }
    assert set(rows_cols) == set(sd), set(rows_cols) ^ set(sd)
    out = {}
    for k, rc in rows_cols.items():
        v = sd[k]
        if rc[0] is not None:
            v = v[rc[0]]
        if len(rc) > 1:
            v = v[:, rc[1]]
        out[k] = v.contiguous()
    return out


def main():
    sys.path.insert(0, REF)
    import text_utils as RT   # the reference's table (prints nothing at import)

    rows = [l.rstrip("\n").split("|") for l in open(os.path.join(REF, "Data", "val_list.txt"), encoding="utf-8").readlines()[:8]]
    dicts = RT.dicts
    sample = {}
    for r in rows[:3]:
        sample[r[1]] = [dicts[c] for c in r[1] if c in dicts]
    json.dump({"symbols": RT.symbols, "sample_ids": sample}, open(os.path.join(GOLD, "textcleaner_vocab.json"), "w"), ensure_ascii=False)

    cells = {}
    for key, nb, idx in (("lj_inference", "Inference_LJSpeech.ipynb", 17), ("lj_LFinference", "Inference_LJSpeech.ipynb", 29),
                         ("libri_inference", "Inference_LibriTTS.ipynb", 16), ("libri_LFinference", "Inference_LibriTTS.ipynb", 42),
                         ("libri_STinference", "Inference_LibriTTS.ipynb", 45)):
        d = json.load(open(os.path.join(REF, "Demo", nb)))
        cells[key] = {"notebook": nb, "cell": idx, "source": "".join(d["cells"][idx]["source"])}
    json.dump(cells, open(os.path.join(GOLD, "notebook_cells.json"), "w"), ensure_ascii=False, indent=1)

    # ---- PL-BERT: a channel slice of the real checkpoint (fp16-rounded on BOTH sides)
    from transformers import AlbertConfig, AlbertModel
    cfg = yaml.safe_load(open(os.path.join(REF, "Utils", "PLBERT", "config.yml")))["model_params"]
    ck = torch.load(os.path.join(REF, "Utils", "PLBERT", "step_1000000.t7"), map_location="cpu", weights_only=True)["net"]
    sd = {}
    for k, v in ck.items():
        name = k[7:] if k.startswith("module.") else k
        if name.startswith("encoder."):
            name = name[8:]
            if name != "embeddings.position_ids" and v.dtype == torch.float32:
                sd[name] = v.half()
    sd = slice_plbert(sd)
    cfg = dict(cfg, **SLICE)
    ref = AlbertModel(AlbertConfig(**cfg)).eval()
    missing, unexpected = ref.load_state_dict({k: v.float() for k, v in sd.items()}, strict=False)
    assert not [m for m in missing if "position_ids" not in m] and not unexpected, (missing, unexpected)
    P = SLICE["max_position_embeddings"]
    toks = [([0] + [dicts[c] for c in r[1] if c in dicts])[:P] for r in rows[:4]]
    N = max(len(t) for t in toks)
    lengths = torch.tensor([len(t) for t in toks])
    tokens = torch.zeros(len(toks), N, dtype=torch.long)
    for i, t in enumerate(toks):
        tokens[i, :len(t)] = torch.tensor(t)
    mask = (torch.arange(N)[None] < lengths[:, None]).int()
    torch.set_num_threads(8)
    with torch.no_grad():
        out = ref(tokens, attention_mask=mask).last_hidden_state
    valid = mask.bool().nonzero()
    pick = valid[torch.randperm(len(valid), generator=torch.Generator().manual_seed(1))[:SLICE_ROWS]]
    pick = pick[torch.argsort(pick[:, 0] * N + pick[:, 1])]
    stats = {k: float(v.float().abs().max()) for k, v in sd.items()}
    print("PL-BERT slice: max |w| per tensor:", {k: round(v, 2) for k, v in sorted(stats.items(), key=lambda kv: -kv[1])[:6]})
    print("output abs max", float(out.abs().max()), "tokens", tuple(tokens.shape), "lengths", lengths.tolist())
    path = os.path.join(GOLD, "plbert_real_slice.npz")
    np.savez_compressed(path, config=np.array(json.dumps(cfg)), tokens=tokens.numpy(), lengths=lengths.numpy(),
                        rows=pick.numpy().astype(np.int64), last_hidden_state_rows=out[pick[:, 0], pick[:, 1]].numpy(),
                        **{"w:" + k: v.numpy() for k, v in sd.items()})
    print("wrote", os.path.getsize(path) / 1e6, "MB")


if __name__ == "__main__":
    main()
