"""Host-side logic on CPU: tokenizer / processor / streamers, the generate() loop contract of the model
object (driven by a scripted engine), the MCTS driver, SelfSim protocol, figure sharding helpers."""
import threading

import pytest
import torch
from PIL import Image, ImageDraw

from scripted_engine import ScriptedEngine


def _model(eos_at=None, max_len=None):
    from detikzify_b200.model import build_processor, preset
    from detikzify_b200.model.modeling import DetikzifyForCausalLM
    cfg = preset("tiny")
    eng = ScriptedEngine(cfg, max_len=max_len, eos_at=eos_at)
    return DetikzifyForCausalLM(cfg, engine=eng), build_processor(cfg), eng


def _figure(size=90):
    im = Image.new("RGB", (size, size + 20), "white")
    d = ImageDraw.Draw(im)
    d.line((10, 10, size - 10, size - 5), fill="black", width=3)
    d.ellipse((20, 30, 50, 60), outline="black")
    return im


# ------------------------------------------------------------------ tokenizer / processor
def test_tokenizer_roundtrip_and_specials():
    from detikzify_b200.model import build_processor, preset
    cfg = preset("tiny")
    proc = build_processor(cfg)
    tok = proc.tokenizer
    text = "\\begin{tikzpicture}\n\\draw (0,0) -- (1,1);\n\\end{tikzpicture}\n"
    ids = tok(text=text)["input_ids"][0]
    assert tok.decode(ids) == text
    assert len(ids) < len(text)                      # multi-character tokens are used
    assert tok.decode([cfg.bos_token_id, 65, cfg.eos_token_id], skip_special_tokens=True) == "A"
    assert proc.image_token == tok.convert_ids_to_tokens(cfg.patch_token_id)
    assert tok.model_max_length == cfg.model_max_length


def test_processor_prompt_layout_and_pixels():
    from detikzify_b200.model import build_processor, preset
    cfg = preset("tiny")
    proc = build_processor(cfg)
    out = proc(images=_figure(), text="ab", return_tensors="pt", text_kwargs={"truncation": True})
    ids = out.input_ids[0].tolist()
    assert ids[: cfg.num_patches] == [cfg.patch_token_id] * cfg.num_patches and ids[cfg.num_patches:] == [97, 98]
    pv = out["pixel_values"]
    assert pv.shape == (1, 3, 56, 56) and pv.dtype == torch.float32
    assert pv.max() <= 1.0 + 1e-6 and pv.min() >= -1.0 - 1e-6 and pv.max() > 0.99   # white background -> +1
    assert set(out.to("cpu").keys()) == {"pixel_values", "input_ids", "attention_mask"}
    with pytest.raises(ValueError):
        proc(text="x", images=None)


def test_streamers_contract():
    from detikzify_b200.util import StreamerList, TextIteratorStreamer, TokenStreamer
    from detikzify_b200.model import build_processor, preset
    st = TokenStreamer()
    st.put(torch.tensor([[1, 2, 3]]))          # prompt is skipped
    st.put(torch.tensor([7]))
    st.put(torch.tensor([8]))
    st.end()
    assert list(st) == [7, 8]
    with pytest.raises(ValueError):
        TokenStreamer().put(torch.zeros(2, 3))
    st2 = TokenStreamer()
    st2.propagate_error(RuntimeError("boom"))
    with pytest.raises(RuntimeError, match="boom"):
        next(st2)
    tok = build_processor(preset("tiny")).tokenizer
    ts = TextIteratorStreamer(tok, skip_prompt=True, skip_special_tokens=True)
    sl = StreamerList([ts])
    sl.put(torch.tensor([[500, 500]]))
    for t in tok.encode("\\draw (0,0);\n"):
        sl.put(torch.tensor([t]))
    sl.end()
    assert "".join(ts) == "\\draw (0,0);\n"


# ------------------------------------------------------------------ generate() contract (scripted engine)
def _prompt(cfg, extra=(65, 66)):
    return torch.tensor([[cfg.patch_token_id] * cfg.num_patches + list(extra)])


def test_generate_streams_prompt_then_tokens_then_end():
    from detikzify_b200.util import TokenStreamer
    model, proc, eng = _model(eos_at=30)
    cfg = model.config
    ids = _prompt(cfg)
    st = TokenStreamer(skip_prompt=False)
    out = model.generate(input_ids=ids, pixel_values=torch.zeros(1, 3, 56, 56), streamer=st,
                         bad_words_ids=[[cfg.image_token_id]], begin_suppress_tokens=[cfg.eos_token_id], max_length=64)
    streamed = list(st)
    assert out.shape[0] == 1 and out[0, : ids.shape[1]].tolist() == ids[0].tolist()
    assert streamed == out[0].tolist()                      # prompt first, then one put per token, then end()
    assert out[0, -1] == cfg.eos_token_id and (out[0, :-1] != cfg.eos_token_id).all()
    assert cfg.image_token_id not in out[0, ids.shape[1]:].tolist()
    assert ("sample", True) in eng.calls                    # EOS suppressed on the first new token only
    assert eng.calls[-1] == ("gen_end",)


def test_generate_max_length_counts_prompt_and_early_returns():
    from detikzify_b200.util import TokenStreamer
    model, proc, eng = _model()
    cfg = model.config
    ids = _prompt(cfg)
    out = model.generate(input_ids=ids, pixel_values=torch.zeros(1, 3, 56, 56), max_length=ids.shape[1] + 9)
    assert out.shape[1] == ids.shape[1] + 9
    steps = [c for c in eng.calls if c == ("gen_step",)]
    assert len(steps) == 8                                   # first token from prefill, n-1 decode steps, no overrun
    st = TokenStreamer()
    out2 = model.generate(input_ids=ids, pixel_values=torch.zeros(1, 3, 56, 56), max_length=ids.shape[1], streamer=st)
    assert out2.shape == ids.shape and list(st) == []        # nothing to do, but the stream is still terminated


def test_generate_abort_within_one_token_and_errors_escape():
    from detikzify_b200.util import ExplicitAbort, TokenStreamer
    model, proc, eng = _model()
    cfg = model.config
    ids = _prompt(cfg)
    ctl = ExplicitAbort()
    seen = []

    class Spy(TokenStreamer):
        def put(self, value):
            super().put(value)
            if value.dim() == 1:
                seen.append(int(value))
                if len(seen) == 5:
                    ctl.abort()
    out = model.generate(input_ids=ids, pixel_values=torch.zeros(1, 3, 56, 56), streamer=Spy(), stopping_criteria=[ctl], max_length=90)
    assert out.shape[1] == ids.shape[1] + 5                  # abort observed right after the 5th token
    bad = torch.tensor([[cfg.patch_token_id] * (cfg.num_patches - 1) + [65, cfg.patch_token_id]])
    with pytest.raises(ValueError, match="consecutive"):
        model.generate(input_ids=bad, pixel_values=torch.zeros(1, 3, 56, 56), max_length=40)
    with pytest.raises(ValueError, match="number of image patch tokens"):
        model.generate(input_ids=bad[:, 1:-1], pixel_values=torch.zeros(1, 3, 56, 56), max_length=40)


def test_generate_reuses_image_features_and_kv_prefix():
    model, proc, eng = _model()
    cfg = model.config
    pix = torch.rand(1, 3, 56, 56)
    ids = _prompt(cfg, extra=(65, 66, 67))
    out = model.generate(input_ids=ids, pixel_values=pix, max_length=ids.shape[1] + 6)
    n_img = sum(1 for c in eng.calls if c[0] == "image_embeds")
    # second call: same figure, prompt = previous output prefix + 2 tokens -> only the suffix is prefilled
    ids2 = torch.cat([out[:, : ids.shape[1] + 3], torch.tensor([[70, 71]])], dim=1)
    eng.calls.clear()
    model.generate(input_ids=ids2, pixel_values=pix.clone(), max_length=ids2.shape[1] + 4)
    pre = [c for c in eng.calls if c[0] == "prefill"][0]
    assert sum(1 for c in eng.calls if c[0] == "image_embeds") == 0 and n_img == 1
    assert pre[2] == ids.shape[1] + 3 and pre[3] == 2        # start_pos = common prefix, 2 new tokens
    # a different figure invalidates both caches
    eng.calls.clear()
    model.generate(input_ids=ids2, pixel_values=torch.rand(1, 3, 56, 56), max_length=ids2.shape[1] + 2)
    pre = [c for c in eng.calls if c[0] == "prefill"][0]
    assert ("image_embeds", (1, 3, 56, 56)) in eng.calls and pre[2] == 0 and pre[3] == ids2.shape[1]


# ------------------------------------------------------------------ MCTS driver
def _fake_renderer():
    def render(code: str):
        if "<t" in code[:0]:
            return None
        im = Image.new("RGB", (64, 64), "white")
        d = ImageDraw.Draw(im)
        for i, ch in enumerate(code[:40]):
            d.point(((ord(ch) * 7 + i) % 64, (ord(ch) * 13 + 3 * i) % 64), fill="black")
        return im
    return render


def test_pipeline_sample_and_mcts_simulate(monkeypatch):
    from detikzify_b200.infer import DetikzifyPipeline, TikzDocument
    model, proc, eng = _model(eos_at=40)
    monkeypatch.setattr(TikzDocument, "backend", staticmethod(_fake_renderer()))
    pipe = DetikzifyPipeline(model, proc, metric="model")
    assert pipe.gen_kwargs["max_length"] == proc.tokenizer.model_max_length and pipe.gen_kwargs["do_sample"]
    doc = pipe.sample(image=_figure())
    assert isinstance(doc, TikzDocument) and ";\n" in doc.code
    results = list(pipe.simulate(image=_figure(), expansions=4))
    assert len(results) == 4
    for score, tikz in results:
        assert -1.0 <= score <= 1.0 + 1e-9 and tikz.is_rasterizable
    with pytest.raises(AssertionError):
        pipe.sample(image=_figure(), text="caption")          # no adapter loaded


def test_mcts_batched_expansions(monkeypatch):
    """rollouts=K: K leaves are expanded per step through ONE generate_batch call (one gen loop over K slots, the common
    prefix shared), rewards come from one batched SelfSim pass, and the tree grows as with sequential expansions."""
    from detikzify_b200.infer import DetikzifyPipeline, TikzDocument
    from detikzify_b200.infer.pipeline import DetikzifyGenerator
    model, proc, eng = _model(eos_at=40)
    monkeypatch.setattr(TikzDocument, "backend", staticmethod(_fake_renderer()))
    pipe = DetikzifyPipeline(model, proc, metric="model")
    gen = DetikzifyGenerator(model=model, processor=proc, image=pipe.load(_figure()), metric=pipe.metric, rollouts=3,
                             **{k: v for k, v in pipe.gen_kwargs.items() if k != "compile_timeout"}, compile_timeout=5)
    eng.calls.clear()
    results = list(gen.simulate(expansions=6))
    assert len(results) == 6 and all(-1.0 <= sc <= 1.0 + 1e-9 and doc.is_rasterizable for sc, doc in results)
    begins = [c for c in eng.calls if c[0] == "gen_begin"]
    assert len(begins) == 2 and all(len(b[1]) == 3 for b in begins)      # two steps of three lock-step rollouts
    vits = [c for c in eng.calls if c[0] == "vit_encode"]
    assert any(c[1][0] == 4 for c in vits)                               # reference + 3 candidate renders in one ViT batch
    root = gen.montecarlo.root_node
    assert root.visits == 6 and root.expanded
    assert gen.montecarlo.stats_expansion_count == 6
    real = [ch for ch in root.children if not ch.is_widen_node]
    assert real and all(ch.parent is root for ch in real)


def test_mcts_tree_growth_and_failed_rollout_memo(monkeypatch):
    from detikzify_b200.infer import DetikzifyGenerator, TikzDocument
    model, proc, eng = _model(eos_at=36)
    monkeypatch.setattr(TikzDocument, "backend", staticmethod(lambda code: None))   # nothing compiles
    gen = DetikzifyGenerator(model, proc, image=_figure(), metric=None, max_length=proc.tokenizer.model_max_length,
                             temperature=0.8, top_p=0.95, top_k=0, do_sample=True)
    outs = [next(gen.simulate(expansions=1)) for _ in range(3)]
    assert all(score <= 0 for score, _ in outs)
    root = gen.montecarlo.root_node
    assert root.visits >= 3 and root.children[0].is_widen_node
    assert gen.newlineinfo[257].num_lines == 1 and gen.newlineinfo[257].trailing


def test_reference_mcts_module_is_drop_in():
    """Our MCTS node updates and scores like the reference's vendored MCTS (recorded from it by
    tests/golden/make_reference_dropin_golden.py) and carries every attribute the reference's node has."""
    import json
    from pathlib import Path
    from detikzify_b200.mcts.node import Node
    ref = json.loads((Path(__file__).resolve().parent / "golden" / "reference_dropin.json").read_text())["mcts_node"]
    mine = Node("s")
    child = Node("c")
    mine.add_child(child)
    child.update_policy_value(1.0)
    child.update_win_value(0.5)
    assert ref["visits"] == mine.visits == 1 and ref["win_value"] == mine.win_value == 0.5
    assert mine.children[0].get_score(mine) == pytest.approx(ref["child_score"])
    assert set(ref["attributes"]) <= set(vars(mine))


def test_dyn_minmax_norm():
    from detikzify_b200.infer import DynMinMaxNorm
    norm = DynMinMaxNorm()
    a = norm(0.2)
    assert a.score == 0                                       # single value -> default
    b = norm(0.8)
    assert a.score == 0.0 and b.score == 1.0                  # lazily re-normalised
    c = norm(0.5) + b + 3
    assert c.score == pytest.approx(0.5 + 1.0 + 3)
    assert (b * 2) == 2.0 and (1 / b) == 1.0


def test_imagesim_protocol():
    from detikzify_b200.evaluate import ImageSim
    model, proc, eng = _model()
    sim = ImageSim.from_detikzify(model, proc)
    sim.update(img1=_figure(), img2=_figure())
    assert sim.compute() == pytest.approx(1.0)
    sim.reset()
    other = Image.new("RGB", (80, 80), "white")
    ImageDraw.Draw(other).rectangle((5, 5, 70, 70), fill="black")
    sim.update(img1=_figure(), img2=other)
    assert sim.compute() < 1.0
    with pytest.raises(NotImplementedError):
        ImageSim(mode="ssim")


def test_imagesim_emd_mode():
    """The v2 models' default SelfSim: 2 tanh(-EMD) + 1 over the patch tokens (reference evaluate/imagesim.py:105-107,121-123).
    The product solves the uniform equal-size transport problem as an assignment problem; here it is held to the transport LP
    itself (what POT's emd2 solves) on random token sets, and run through the public protocol on the scripted tower."""
    import math
    import numpy as np
    from scipy.optimize import linprog
    from detikzify_b200.evaluate import ImageSim
    g = torch.Generator().manual_seed(7)
    for n, d in ((5, 8), (12, 16), (16, 6)):
        f1, f2 = torch.randn(n, d, generator=g), torch.randn(n, d, generator=g)
        a, b = f1.double() / f1.double().norm(dim=1, keepdim=True), f2.double() / f2.double().norm(dim=1, keepdim=True)
        M = (1.0 - a @ b.T).numpy()
        A_eq = np.zeros((2 * n, n * n))
        for i in range(n):
            A_eq[i, i * n:(i + 1) * n] = 1.0
            A_eq[n + i, i::n] = 1.0
        res = linprog(M.reshape(-1), A_eq=A_eq, b_eq=np.full(2 * n, 1.0 / n), bounds=(0, None), method="highs")
        assert res.status == 0
        assert ImageSim._emd_similarity(f1, f2) == pytest.approx(2 * math.tanh(-res.fun) + 1, abs=1e-9)
    assert ImageSim._emd_similarity(f1, f1) == pytest.approx(1.0, abs=1e-12)
    with pytest.raises(ValueError):
        ImageSim._emd_similarity(f1, f2[:3])
    model, proc, eng = _model()
    sim = ImageSim.from_detikzify(model, proc, mode="emd")
    assert str(sim) == "ImageSim (EMD)"
    other = Image.new("RGB", (80, 80), "white")
    ImageDraw.Draw(other).rectangle((5, 5, 70, 70), fill="black")
    same, diff = sim.get_similarity(_figure(), _figure()), sim.get_similarity(_figure(), other)
    assert same == pytest.approx(1.0) and -1.0 < diff < 1.0
    assert sim.get_similarities([_figure(), other], _figure()) == pytest.approx([same, diff])


def test_pooling_mode_follows_the_model_generation():
    """v1 configs pool with "cos" (v1/configuration_detikzify.py:11-13); the v2 config has no pooling_mode, so the reference's
    ImageSim.from_detikzify falls back to "emd" (evaluate/imagesim.py:64)."""
    from detikzify_b200.model.configuration import preset
    assert preset("tiny").pooling_mode == "cos" and preset("nllg/detikzify-ds-1.3b").pooling_mode == "cos"
    assert preset("tiny-v2").pooling_mode == "emd" and preset("nllg/detikzify-v2-8b").pooling_mode == "emd"


def test_shard_and_interleave():
    from detikzify_b200.parallel import interleave, shard
    items = list(range(11))
    chunks = [shard(items, r, 4) for r in range(4)]
    assert chunks[1] == [1, 5, 9] and interleave(chunks) == items


# ------------------------------------------------------------------ batched generation (extension)
def test_generate_batch_equals_separate_generate_calls():
    """N sequences decoded in lock-step give what N batch-1 generate() calls give (same processors, own EOS / max_length
    per sequence), with one gen loop over all slots and every KV slot handed back."""
    model, proc, eng = _model(eos_at=40)
    pix = torch.rand(1, 3, 56, 56)
    prompts = []
    for extra in (0, 3, 9):
        enc = proc(images=_figure(), text=None, return_tensors="pt")
        prompts.append(torch.cat([enc.input_ids[0], torch.arange(40, 40 + extra)]))
    singles = [model.generate(input_ids=p[None], pixel_values=pix, max_length=60, do_sample=False,
                              bad_words_ids=[[model.config.image_token_id]], begin_suppress_tokens=[model.config.eos_token_id])[0]
               for p in prompts]
    eng.calls.clear()
    free_before = set(eng._slots)
    outs = model.generate_batch(prompts, pixel_values=pix, max_length=60, do_sample=False,
                                bad_words_ids=[[model.config.image_token_id]], begin_suppress_tokens=[model.config.eos_token_id])
    assert [o.tolist() for o in outs] == [s.tolist() for s in singles]
    assert len({len(o) - len(p) for o, p in zip(outs, prompts)}) == 3   # they really stopped at different steps
    begins = [c for c in eng.calls if c[0] == "gen_begin"]
    assert len(begins) == 1 and len(begins[0][1]) == 3            # ONE loop over the three slots
    assert sum(1 for c in eng.calls if c[0] == "image_embeds") == 1
    assert set(eng._slots) == free_before                          # slots released


def test_generate_batch_shared_prefix_streamers_and_per_sequence_stop():
    """Rollouts of one figure: the common prefix (image span + tree path) is prefilled once and lent to every sequence
    (seq_share), each sequence prefills only its suffix; every sequence feeds its own streamer (prompt once, tokens one by
    one, end()) and obeys its own stopping criterion. Tokens equal separate generate() calls."""
    from detikzify_b200.util import TokenStreamer
    model, proc, eng = _model(eos_at=None)
    pix = torch.rand(1, 3, 56, 56)
    enc = proc(images=_figure(), text=None, return_tensors="pt")
    path = torch.arange(40, 62)                                       # 22 shared path tokens after the 5 image tokens
    prompts = [torch.cat([enc.input_ids[0], path, torch.arange(70 + 10 * i, 70 + 10 * i + 2 + i)]) for i in range(3)]
    kw = dict(max_length=70, do_sample=False, bad_words_ids=[[model.config.image_token_id]],
              begin_suppress_tokens=[model.config.eos_token_id])
    singles = [model.generate(input_ids=p[None], pixel_values=pix, **kw)[0] for p in prompts]
    eng.calls.clear()
    free_before = set(eng._slots)
    streamers = [TokenStreamer(skip_prompt=True), None, TokenStreamer(skip_prompt=False)]
    stop_after = 4                                                    # sequence 1 stops after 4 new tokens
    crit = [[], [lambda ids, scores: ids.shape[1] >= len(prompts[1]) + stop_after], []]
    outs = model.generate_batch(prompts, pixel_values=pix, streamers=streamers, stopping_criteria=crit, **kw)
    assert outs[0].tolist() == singles[0].tolist() and outs[2].tolist() == singles[2].tolist()
    assert outs[1].tolist() == singles[1].tolist()[: len(prompts[1]) + stop_after]
    assert list(streamers[0]) == outs[0].tolist()[len(prompts[0]):]
    assert list(streamers[2]) == outs[2].tolist()                    # skip_prompt=False: prompt tokens first
    shares = [c for c in eng.calls if c[0] == "seq_share"]
    lcp = 5 + 22
    assert len(shares) == 3 and all(c[3] == lcp for c in shares) and len({c[1] for c in shares}) == 1
    pre = [c for c in eng.calls if c[0] == "prefill"]
    assert pre[0][2:4] == (0, lcp) and pre[0][4]                      # the shared head, with the image, once
    assert [c[2] for c in pre[1:]] == [lcp] * 3 and [c[3] for c in pre[1:]] == [2, 3, 4] and not any(c[4] for c in pre[1:])
    assert set(eng._slots) == free_before


def test_generate_batch_limits_and_validation():
    model, proc, eng = _model()
    enc = proc(images=_figure(), text=None, return_tensors="pt")
    ids = enc.input_ids[0]
    pix2 = torch.rand(2, 3, 56, 56)
    outs = model.generate_batch([ids, ids], pixel_values=pix2, max_new_tokens=5)
    assert [len(o) for o in outs] == [len(ids) + 5] * 2
    assert ("image_embeds", (2, 3, 56, 56)) in eng.calls
    assert model.generate_batch([], pixel_values=None) == []
    short = model.generate_batch([ids], pixel_values=pix2[:1], max_length=len(ids))      # prompt already at max_length
    assert short[0].tolist() == ids.tolist()
    with pytest.raises(ValueError):
        model.generate_batch([ids[1:]], pixel_values=pix2[:1], max_new_tokens=3)         # wrong number of patch tokens
    with pytest.raises(ValueError):
        model.generate_batch([ids, ids, ids], pixel_values=pix2, max_new_tokens=3)       # 2 images for 3 sequences


def test_pipeline_sample_batch(monkeypatch):
    from detikzify_b200.infer import DetikzifyPipeline, TikzDocument
    model, proc, eng = _model(eos_at=40)
    monkeypatch.setattr(TikzDocument, "backend", staticmethod(_fake_renderer()))
    pipe = DetikzifyPipeline(model, proc, metric="fast")
    docs = pipe.sample_batch([_figure(), _figure(70)], samples_per_image=2)
    assert len(docs) == 4 and all(isinstance(d, TikzDocument) and d.code for d in docs)
    begins = [c for c in eng.calls if c[0] == "gen_begin"]
    assert len(begins) == 1 and len(begins[0][1]) == 4            # one lock-step loop over the four sequences
    assert ("image_embeds", (4, 3, 56, 56)) in eng.calls
    assert eng.last_sampling["do_sample"] and abs(eng.last_sampling["temperature"] - 0.8) < 1e-9


# ------------------------------------------------------------------ KV prefix cache over several slots
def _prefilled(eng):
    return sum(c[3] for c in eng.calls if c[0] == "prefill")


def test_prefix_cache_over_slots_avoids_thrashing():
    """Alternating between two branches of a search tree: with one slot every switch re-prefills the branch, with a slot
    cache only the new suffix is prefilled (the shared prefix is forked). Outputs are identical either way."""
    from detikzify_b200.model import build_processor, preset
    from detikzify_b200.model.modeling import DetikzifyForCausalLM
    cfg = preset("tiny")
    proc = build_processor(cfg)
    base = proc(images=_figure(), text=None, return_tensors="pt").input_ids[0]
    pix = torch.rand(1, 3, 56, 56)
    A = torch.cat([base, torch.arange(40, 60)])
    B = torch.cat([base, torch.arange(70, 90)])
    A2 = torch.cat([A, torch.arange(100, 104)])
    B2 = torch.cat([B, torch.arange(110, 114)])
    A3 = torch.cat([A[:-5], torch.arange(120, 124)])       # leaves A's content in the middle
    seq = [A, B, A2, B2, A3, A2]
    runs = {}
    for slots in (1, 4):
        eng = ScriptedEngine(cfg, max_len=90)
        model = DetikzifyForCausalLM(cfg, engine=eng, prefix_slots=slots)
        outs = [model.generate(input_ids=p[None], pixel_values=pix, max_new_tokens=6)[0].tolist() for p in seq]
        runs[slots] = (outs, _prefilled(eng), [c for c in eng.calls if c[0] == "seq_fork"])
    assert runs[1][0] == runs[4][0]                          # same results
    assert not runs[1][2] and runs[4][2]                     # forks only with the cache
    assert runs[4][1] < 0.6 * runs[1][1], (runs[4][1], runs[1][1])
    # every fork copies exactly the shared prefix and never splits the image span
    P = cfg.num_patches
    for _, src, dst, length in runs[4][2]:
        assert src != dst and (length >= P or length == 0)


def test_prefix_cache_invalidated_by_new_image_and_bounded_by_engine_slots():
    from detikzify_b200.model import build_processor, preset
    from detikzify_b200.model.modeling import DetikzifyForCausalLM
    cfg = preset("tiny")
    proc = build_processor(cfg)
    ids = proc(images=_figure(), text=None, return_tensors="pt").input_ids
    eng = ScriptedEngine(cfg, max_len=90)
    model = DetikzifyForCausalLM(cfg, engine=eng, prefix_slots=3)
    model.generate(input_ids=ids, pixel_values=torch.rand(1, 3, 56, 56), max_new_tokens=4)
    n0 = _prefilled(eng)
    model.generate(input_ids=ids, pixel_values=torch.rand(1, 3, 56, 56), max_new_tokens=4)   # another figure
    assert _prefilled(eng) - n0 == ids.shape[1]              # nothing reused across images
    assert len(model._kv) <= 3
    # the engine refusing further slots only disables growth
    eng.seq_alloc = lambda: (_ for _ in ()).throw(RuntimeError("no free KV slot"))
    other = torch.cat([ids[0], torch.arange(50, 55)])[None]
    out = model.generate(input_ids=other, pixel_values=None, max_new_tokens=3)
    assert out.shape[1] == other.shape[1] + 3


# ------------------------------------------------------------------ checkpoint directory loading (host side)
def test_checkpoint_directory_config_and_state_dict(tmp_path):
    """load() on a local directory: config.json decides the shape (v1 flat / v2 nested), v2 parameter names map onto the
    canonical ones, and a v1 checkpoint without a vision tower asks for one instead of failing with a KeyError."""
    import json
    from safetensors.torch import save_file
    from detikzify_b200.model import _load_safetensors_dir
    from detikzify_b200.model.configuration import config_from_dict, preset
    from detikzify_b200.model.weights import random_init, to_v2_state_dict
    cfg = preset("tiny-v2")
    sd = random_init(cfg)
    d = tmp_path / "v2"
    d.mkdir()
    save_file({k: v.contiguous() for k, v in to_v2_state_dict(sd).items()}, str(d / "model.safetensors"))
    text = dict(hidden_size=cfg.hidden_size, intermediate_size=cfg.intermediate_size, num_hidden_layers=cfg.num_hidden_layers,
                num_attention_heads=cfg.num_attention_heads, num_key_value_heads=cfg.num_key_value_heads, head_dim=128,
                vocab_size=cfg.vocab_size, rms_norm_eps=1e-5, rope_theta=500000.0, bos_token_id=600, eos_token_id=601, pad_token_id=604,
                rope_scaling=dict(rope_type="llama3", factor=8.0, low_freq_factor=1.0, high_freq_factor=4.0, original_max_position_embeddings=64))
    (d / "config.json").write_text(json.dumps(dict(image_token_id=605, concat_factor=3, text_config=text,
                                                   vision_config=cfg.vision_config.to_dict())))
    got = config_from_dict(json.loads((d / "config.json").read_text()), name=str(d))
    for k in ("hidden_size", "num_key_value_heads", "rope_type", "rope_original_max_position", "patch_token_id", "projector_bias", "num_patches"):
        assert getattr(got, k) == getattr(cfg, k), k
    loaded = _load_safetensors_dir(str(d))
    assert set(loaded) == set(sd) and all(torch.equal(loaded[k], sd[k]) for k in sd)
    # v1: decoder-only checkpoint -> explicit request for the tower
    v1 = tmp_path / "v1"
    v1.mkdir()
    cfg1 = preset("tiny")
    sd1 = {k: v for k, v in random_init(cfg1).items() if "vision_model" not in k}
    save_file({k: v.contiguous() for k, v in sd1.items()}, str(v1 / "model.safetensors"))
    with pytest.raises(FileNotFoundError, match="vision_tower"):
        _load_safetensors_dir(str(v1))


def test_pil_resample_restatement_is_bit_exact():
    """The fixed-point bicubic resize the device kernels implement (model/processing.py::pil_resample_reference, taps from
    pil_resample_coeffs) equals Pillow's ``Image.resize(BICUBIC)`` bit for bit, up- and down-scaling, non-square inputs."""
    import numpy as np
    from detikzify_b200.model.processing import pil_resample_reference
    rng = np.random.default_rng(1)
    for h, w, S in [(300, 300, 56), (56, 56, 56), (61, 147, 56), (40, 40, 96), (700, 433, 384)]:
        arr = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        ref = np.asarray(Image.fromarray(arr).resize((S, S), resample=Image.Resampling.BICUBIC))
        assert np.array_equal(pil_resample_reference(arr, S), ref), (h, w, S)
