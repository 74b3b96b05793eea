"""
Drop-in boundary (SURVEY.md §8b), checked against recordings of the original project: its own inference driver
(detikzify/infer/generate.py: DetikzifyGenerator, DetikzifyPipeline, WideNode, rollout streaming), its vendored MCTS, its
SelfSim reward (evaluate/imagesim.py) and its v1 image processor were run on the objects ``detikzify_b200`` returns (model
with ``generate``, processor, tokenizer), with the scripted engine standing in for the GPU, by
``tests/golden/make_reference_dropin_golden.py``. What they did — the engine calls and generation kwargs of a sample, the
programs, scores and tree sizes of MCTS runs, the SelfSim values, the pixels they computed — is stored in
``tests/golden/reference_dropin.*``.
Here our own driver, MCTS, SelfSim and processor run on the same objects and must do the same.

The recordings were taken with the TeX toolchain stubbed (every program "compiles" into a white 32x32 page); our
``TikzDocument`` gets the same stand-in renderer here.
"""
import json
from pathlib import Path

import numpy as np
import pytest
import torch
from PIL import Image, ImageDraw

from scripted_engine import ScriptedEngine

GOLDEN = Path(__file__).resolve().parent / "golden"


@pytest.fixture(scope="module")
def gold():
    return json.loads((GOLDEN / "reference_dropin.json").read_text()), np.load(GOLDEN / "reference_dropin.npz")


@pytest.fixture()
def compiles(monkeypatch):
    """The stand-in TeX toolchain of the recordings: every program compiles into a white 32x32 page."""
    from detikzify_b200.infer import TikzDocument
    monkeypatch.setattr(TikzDocument, "backend", staticmethod(lambda code: Image.new("RGB", (32, 32), "white")))


def _ours(eos_at=40):
    from detikzify_b200.model import build_processor, preset
    from detikzify_b200.model.modeling import DetikzifyForCausalLM
    cfg = preset("tiny")
    eng = ScriptedEngine(cfg, eos_at=eos_at)
    return DetikzifyForCausalLM(cfg, engine=eng), build_processor(cfg), eng


def _figure(size=90):
    im = Image.new("RGB", (size, size + 20), "white")
    d = ImageDraw.Draw(im)
    d.line((10, 10, size - 10, size - 5), fill="black", width=3)
    d.ellipse((20, 30, 50, 60), outline="black")
    return im


def _other():
    im = Image.new("RGB", (80, 80), "white")
    ImageDraw.Draw(im).ellipse((10, 10, 60, 70), outline="black", width=4)
    return im


def _preprocess_inputs():
    rng = np.random.default_rng(3)
    return [_figure(90), _figure(384).resize((384, 384)), Image.fromarray(rng.integers(0, 255, (200, 311, 3), dtype=np.uint8))]


# the recorded form of engine calls, documents and sampler arguments (shared with the script that records the original project)
def calls_json(calls):
    return json.loads(json.dumps(calls))


def doc_json(doc):
    return {"code": doc.code, "compiled_with_errors": bool(doc.compiled_with_errors), "rasterizable": bool(doc.is_rasterizable)}


def sampling_json(kw):
    """The sampler arguments generate() was given; the RNG seed is drawn per call and is left out."""
    return {k: v for k, v in kw.items() if k != "seed"}


def test_reference_pipeline_sample_runs_on_our_model(gold, compiles):
    from detikzify_b200.infer import DetikzifyPipeline
    ref = gold[0]["sample"]
    model, proc, eng = _ours(eos_at=30)
    pipe = DetikzifyPipeline(model=model, processor=proc, metric="fast")
    assert {k: pipe.gen_kwargs.get(k) for k in ref["gen_kwargs"]} == ref["gen_kwargs"]
    assert pipe.gen_kwargs["max_length"] == proc.tokenizer.model_max_length and pipe.gen_kwargs["do_sample"] is True
    doc = pipe.sample(image=_figure())
    assert doc_json(doc) == ref["doc"] and len(doc.code) > 0
    # the same generation kwargs reach generate() (reference infer/generate.py:218-227), through the same engine calls
    kw = eng.last_sampling
    assert sampling_json(kw) == ref["sampling"]
    assert kw["bad_token"] == model.config.image_token_id and kw["begin_suppress_token"] == model.config.text_config.eos_token_id
    assert kw["do_sample"] and abs(kw["temperature"] - 0.8) < 1e-6 and abs(kw["top_p"] - 0.95) < 1e-6
    assert calls_json(eng.calls) == ref["calls"]


def test_reference_mcts_simulate_runs_on_our_model(gold, compiles):
    from detikzify_b200.infer import DetikzifyPipeline
    ref = gold[0]["simulate_fast"]
    model, proc, eng = _ours(eos_at=36)
    pipe = DetikzifyPipeline(model=model, processor=proc, metric="fast")
    results = list(pipe.simulate(image=_figure(), expansions=4))
    assert len(results) == 4 and all(score == 1 for score, _ in results)   # scorable - compiled_with_errors
    # later expansions start wherever the tree search (random among equal scores) goes; the first one is from the root
    assert [s for s, _ in results] == ref["scores"] and doc_json(results[0][1]) == ref["first_doc"]
    # rollouts went through the TokenStreamer + stopping-criteria path and our streaming contract
    assert sum(1 for c in eng.calls if c[0] == "gen_begin") >= 4


def test_reference_generator_abort_and_tree(gold, compiles):
    from detikzify_b200.infer.pipeline import DetikzifyGenerator
    ref = gold[0]["generator_tree"]
    model, proc, eng = _ours(eos_at=60)
    gen = DetikzifyGenerator(model=model, processor=proc, image=_figure(), metric=None, max_length=proc.tokenizer.model_max_length,
                             temperature=0.8, top_p=0.95, top_k=0, do_sample=True)
    out = [next(gen.simulate(expansions=1)) for _ in range(2)]
    root = gen.montecarlo.root_node
    assert root.visits >= 2 and root.children and root.children[0].is_widen_node
    assert all(score == 1 for score, _ in out)
    assert [s for s, _ in out] == ref["scores"] and doc_json(out[0][1]) == ref["first_doc"]
    assert root.visits == ref["root_visits"] and root.children[0].is_widen_node == ref["first_child_widen"]
    # newline bookkeeping works with our tokenizer (vocab / decode protocol) as the reference's did
    assert gen.newlineinfo and {str(k): [v.num_lines, v.trailing] for k, v in sorted(gen.newlineinfo.items())} == ref["newlineinfo"]


def test_reference_selfsim_metric_runs_on_our_vision_model(gold, compiles):
    """metric="model": the SelfSim reward wraps OUR model.model.vision_model / image processor and is computed from
    pooler_output (reference evaluate/imagesim.py:60-125); MCTS then min-max-normalises it."""
    from detikzify_b200.infer import DetikzifyPipeline
    ref = gold[0]["simulate_selfsim"]
    model, proc, eng = _ours(eos_at=36)
    pipe = DetikzifyPipeline(model=model, processor=proc, metric="model")
    assert type(pipe.metric).__name__ == "ImageSim" and pipe.metric.mode == ref["mode"] == "cos"
    pipe.metric.update(img1=_figure(), img2=_figure())
    assert pipe.metric.compute() == pytest.approx(ref["same_figure"]) == pytest.approx(1.0)   # identical figures -> cosine 1
    pipe.metric.reset()
    results = list(pipe.simulate(image=_figure(), expansions=3))
    assert len(results) == 3 and all(-1.0 <= score <= 1.0 + 1e-9 for score, _ in results)
    assert len(ref["scores"]) == 3 and doc_json(results[0][1]) == ref["first_doc"]
    assert any(c[0] == "vit_encode" for c in eng.calls)


def test_reference_emd_selfsim_agrees_with_ours(gold):
    """The v2 default reward: the reference's ImageSim in "emd" mode (evaluate/imagesim.py:105-107,121-123; POT's emd2
    restated as the transport LP) and ours (assignment solver) on the same vision model object and image processor."""
    from detikzify_b200.evaluate.imagesim import ImageSim as Ours
    ref, arrays = gold[0]["emd"], gold[1]
    model, proc, eng = _ours(eos_at=36)
    ours = Ours.from_detikzify(model, proc, mode="emd")
    # the reference object fed bf16 pixels (its .to(device, dtype)), ours fp32: compare the solvers on the SAME patch tokens ...
    f1, f2 = torch.from_numpy(arrays["emd_f1"]), torch.from_numpy(arrays["emd_f2"])
    a = ref["similarity"]
    assert f1.ndim == 2 and a == pytest.approx(Ours._emd_similarity(f1, f2), abs=1e-9) and -1.0 < a < 1.0
    # ... and the two end-to-end paths within the bf16 rounding of the inputs
    assert a == pytest.approx(ours.get_similarity(_figure(), _other()), abs=5e-2)
    assert ref["same_figure"] == pytest.approx(1.0, abs=1e-9)
    assert ours.get_similarity(_figure(), _figure()) == pytest.approx(1.0, abs=1e-9)


def test_image_processor_matches_reference_preprocess(gold):
    """§8 row a1: our host-side DetikzifyImageProcessor against the reference's own class
    (detikzify/model/v1/processing_detikzify.py:162-253), built from the dict its ``from_pretrained`` assembles (:104-117)
    with timm's published config of vit_so400m_patch14_siglip_384: input 3x384x384, mean = std = 0.5, bicubic."""
    from detikzify_b200.model.processing import DetikzifyImageProcessor
    ref, arrays = gold[0]["image_processor"], gold[1]
    ours = DetikzifyImageProcessor(size=384)
    assert ref["size"] == ours.size and ref["image_mean"] == ours.image_mean and ref["image_std"] == ours.image_std
    assert ref["resample"] == ours.resample == 3 and abs(ref["rescale_factor"] - ours.rescale_factor) < 1e-12
    for i, im in enumerate(_preprocess_inputs()):
        a = (torch.from_numpy(arrays[f"pixels_{i}"]).double() / 255 - 0.5) / 0.5
        b = ours(im, return_tensors="pt")["pixel_values"]
        assert a.shape == b.shape == (1, 3, 384, 384) and b.dtype == torch.float32
        assert (a - b.double()).abs().max().item() < 1e-6
