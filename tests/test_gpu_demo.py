"""GPU tier: the notebook-level boundary.  The inference cells of the reference's Demo notebooks are exec()'d VERBATIM
(source text from tests/golden/notebook_cells.json, extracted from the unmodified notebooks) over this package's
build_model() container -- same globals as the notebooks: model, sampler, textclenaer, global_phonemizer, word_tokenize,
device, length_to_mask -- and compared with styletts2_b200.demo's entry points (the Synthesizer engine: device-side
durations, gather alignment, no host loop).  PL-BERT runs with a channel slice of the REAL bundled checkpoint (two of its
twelve heads, its extreme values kept; fp16-rounded fixture written by oracle/make_golden_demo.py)."""
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from util import GOLD, maxdiff, record

D = "cuda:0"


def _texts():
    """two short IPA phoneme strings: the first words of two Data/val_list.txt rows (fixture)"""
    rows = list(json.load(open(os.path.join(GOLD, "textcleaner_vocab.json"), encoding="utf-8"))["sample_ids"])
    return " ".join(rows[0].split()[:5]) + " .", " ".join(rows[1].split()[:6]) + " ."


def _real_plbert():
    from styletts2_b200.plbert import PLBert
    g = np.load(os.path.join(GOLD, "plbert_real_slice.npz"))
    sd = {k[2:]: torch.from_numpy(g[k]).float() for k in g.files if k.startswith("w:")}
    bert = PLBert(**json.loads(str(g["config"]))).to(D).eval()
    missing, unexpected = bert.load_state_dict(sd, strict=False)
    assert not missing, missing
    return bert, g, sd


_NB = {}


def _notebook(model_name):
    if model_name in _NB:
        return _NB[model_name]
    from styletts2_b200.configs import MODEL_CFGS
    from styletts2_b200.demo import bind
    from styletts2_b200.models import build_model, load_keyed_weights, recursive_munch
    bert, _, _ = _real_plbert()
    params = recursive_munch(MODEL_CFGS[model_name])
    model = build_model(params, bert=bert)
    for k in model:
        model[k].to(D).eval()
    load_keyed_weights(model)
    nb = bind(model, MODEL_CFGS[model_name], D)
    glb = dict(torch=torch, model=model, sampler=nb.sampler, textclenaer=nb.textclenaer, global_phonemizer=nb.global_phonemizer,
               word_tokenize=nb.word_tokenize, device=D, length_to_mask=nb.length_to_mask, model_params=params)
    cells = json.load(open(os.path.join(GOLD, "notebook_cells.json"), encoding="utf-8"))
    _NB[model_name] = (nb, glb, cells)
    return _NB[model_name]


def _cell_fn(glb, cells, key, name):
    ns = dict(glb)
    exec(compile(cells[key]["source"], f"<{cells[key]['notebook']}#cell{cells[key]['cell']}>", "exec"), ns)
    return ns[name]


def _seed():
    from styletts2_b200 import ops
    ops.manual_seed(1234)
    torch.manual_seed(99)
    return ops


def test_plbert_with_the_real_checkpoint_matches_transformers():
    """Row f1 on the real weight distribution (key.bias up to 13, LayerNorm gains ~3): also a range check of the fp16
    two-plane GEMM (|x| < 65504) that the default-init test cannot give.  The stored rows are transformers.AlbertModel's
    output recorded with the fixture; every other valid row is checked against the installed transformers."""
    from transformers import AlbertConfig, AlbertModel
    bert, g, sd = _real_plbert()
    tokens, lengths = torch.from_numpy(g["tokens"]), torch.from_numpy(g["lengths"])
    N = tokens.shape[1]
    mask = (torch.arange(N)[None] < lengths[:, None])
    with torch.no_grad():
        got = bert(tokens.to(D), attention_mask=mask.int().to(D)).cpu()
    assert torch.isfinite(got[mask]).all()
    rows = torch.from_numpy(g["rows"])
    want_rows = torch.from_numpy(g["last_hidden_state_rows"])
    e = float((got[rows[:, 0], rows[:, 1]] - want_rows).abs().max()) / float(want_rows.abs().max())
    ref = AlbertModel(AlbertConfig(**json.loads(str(g["config"])))).eval()
    ref.load_state_dict(sd, strict=False)
    with torch.no_grad():
        want = ref(tokens, attention_mask=mask.int()).last_hidden_state
    assert float((want[rows[:, 0], rows[:, 1]] - want_rows).abs().max()) <= 1e-5 * float(want_rows.abs().max())
    e_all = float((got - want)[mask].abs().max()) / float(want[mask].abs().max())
    record("plbert_real_checkpoint", rel_err=e, rel_err_all_rows=e_all, rows=int(mask.sum()))
    assert e < 5e-5, e
    assert e_all < 5e-5, e_all


def test_lj_inference_cell_verbatim_equals_demo_inference():
    nb, glb, cells = _notebook("ljspeech")
    cell_inference = _cell_fn(glb, cells, "lj_inference", "inference")
    text = _texts()[0]
    noise = torch.randn(1, 1, 256, generator=torch.Generator().manual_seed(5)).to(D)
    ops = _seed()
    ops.rng_advance(torch.device(D))            # Synthesizer.synthesize starts a new draw epoch per call
    w_cell = cell_inference(text, noise, diffusion_steps=5, embedding_scale=1)
    _seed()
    w_ours = nb.inference(text, noise, diffusion_steps=5, embedding_scale=1)
    assert w_cell.shape == w_ours.shape and w_cell.dtype == np.float32
    d = float(np.abs(w_cell - w_ours).max())
    record("demo_lj_inference_vs_cell", wav_maxabs=d, samples=int(w_ours.shape[0]))
    assert d <= 1e-5, d


def test_lj_LFinference_cell_verbatim_has_no_last_token_increment():
    nb, glb, cells = _notebook("ljspeech")
    cell_lf = _cell_fn(glb, cells, "lj_LFinference", "LFinference")
    noise = torch.randn(1, 1, 256, generator=torch.Generator().manual_seed(6)).to(D)
    s_prev = None
    for text in _texts():
        ops = _seed()
        ops.rng_advance(torch.device(D))
        w_cell, s_cell = cell_lf(text, s_prev, noise, alpha=0.7, diffusion_steps=3, embedding_scale=1)
        _seed()
        w_ours, s_ours = nb.LFinference(text, s_prev, noise, alpha=0.7, diffusion_steps=3, embedding_scale=1)
        assert w_cell.shape == w_ours.shape          # same total duration: no `pred_dur[-1] += 5` in cell 29
        assert float(np.abs(w_cell - w_ours).max()) <= 1e-5
        assert maxdiff(s_cell, s_ours) <= 1e-6
        s_prev = s_ours


@pytest.mark.parametrize("which", ["inference", "LFinference", "STinference"])
def test_libri_cells_verbatim_equal_demo(which):
    nb, glb, cells = _notebook("libritts")
    ta, tb = _texts()
    ref_s = (torch.randn(1, 256, generator=torch.Generator().manual_seed(8)) * 0.3).to(D)
    fn_cell = _cell_fn(glb, cells, "libri_" + which, which)
    fn_ours = nb[which]
    if which == "inference":
        args, kw = (ta, ref_s), dict(alpha=0.3, beta=0.7, diffusion_steps=4, embedding_scale=1)
    elif which == "LFinference":
        s_prev = (torch.randn(1, 256, generator=torch.Generator().manual_seed(9)) * 0.3).to(D)
        args, kw = (tb, s_prev, ref_s), dict(alpha=0.3, beta=0.7, t=0.7, diffusion_steps=3, embedding_scale=1)
    else:
        args, kw = (ta, ref_s, tb), dict(alpha=0.3, beta=0.7, diffusion_steps=3, embedding_scale=1)
    ops = _seed()
    ops.rng_advance(torch.device(D))
    r_cell = fn_cell(*args, **kw)
    _seed()
    r_ours = fn_ours(*args, **kw)
    w_cell, w_ours = (r_cell[0], r_ours[0]) if which == "LFinference" else (r_cell, r_ours)
    assert w_cell.shape == w_ours.shape              # incl. the [..., :-50] / [..., :-100] trims
    d = float(np.abs(w_cell - w_ours).max())
    record("demo_libri_vs_cell", which=which, wav_maxabs=d, samples=int(w_ours.shape[0]))
    assert d <= 1e-5, d
    if which == "LFinference":
        assert maxdiff(r_cell[1], r_ours[1]) <= 1e-6
