"""
Writes ``reference_dropin.json`` and ``reference_dropin.npz``: what the original DeTikZify project's own host code (its
inference driver ``detikzify/infer/generate.py``, the vendored MCTS ``detikzify/mcts``, the SelfSim reward
``detikzify/evaluate/imagesim.py`` and the v1 image processor ``detikzify/model/v1/processing_detikzify.py``) does when it
runs on the objects ``detikzify_b200`` returns, with ``tests/scripted_engine.py`` standing in for the GPU.
``tests/test_cpu_reference_dropin.py`` holds our own driver, MCTS, SelfSim and processor to these recordings.

The original modules are executed from a checkout of the original project, never copied. Stubbed because they are absent
offline: torchmetrics (the slice of ``Metric`` that ImageSim uses, and ``pairwise_cosine_similarity``), the TeX toolchain
(``infer/tikz.py`` -> a TikzDocument that "compiles" everything into a white 32x32 page), ``util/image.py`` (two small PIL
helpers), ``model/adapter`` (``has_adapter`` -> False), POT's ``emd2`` (restated as the transport LP) and, for the image
processor, timm's published data config of vit_so400m_patch14_siglip_384 (input 3x384x384, mean = std = 0.5, bicubic).

Run:  python tests/golden/make_reference_dropin_golden.py <checkout of the original project>
"""
from __future__ import annotations

import importlib.util
import json
import sys
import types
from pathlib import Path

import numpy as np
import torch
from PIL import Image

HERE = Path(__file__).resolve().parent
sys.path[:0] = [str(HERE.parent.parent), str(HERE.parent)]

from test_cpu_reference_dropin import (_figure, _other, _ours, _preprocess_inputs, calls_json, doc_json,  # noqa: E402
                                       sampling_json)


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def load_reference_infer(ref: Path):
    """The original ``detikzify.infer.generate`` with its own MCTS, util and ImageSim modules, on the stubs above."""
    tm = types.ModuleType("torchmetrics")
    sys.modules["torchmetrics"] = tm
    for pkg in ("detikzify", "detikzify.infer", "detikzify.mcts", "detikzify.util", "detikzify.model", "detikzify.evaluate"):
        m = types.ModuleType(pkg)
        m.__path__ = []
        sys.modules[pkg] = m
    _load("detikzify.mcts.node", ref / "mcts/node.py")
    _load("detikzify.mcts.montecarlo", ref / "mcts/montecarlo.py")
    fn = _load("detikzify.util.functools", ref / "util/functools.py")
    gn = _load("detikzify.util.generation", ref / "util/generation.py")
    util = sys.modules["detikzify.util"]
    for mod in (fn, gn):
        for k, v in vars(mod).items():
            if not k.startswith("_"):
                setattr(util, k, v)
    util.load = lambda image: image.convert("RGB") if isinstance(image, Image.Image) else Image.open(image).convert("RGB")

    def expand(image, size, do_trim=False):
        canvas = Image.new("RGB", (size, size), "white")
        canvas.paste(image, ((size - image.width) // 2, (size - image.height) // 2))
        return canvas
    util.expand = expand
    adapter = types.ModuleType("detikzify.model.adapter")
    adapter.has_adapter = lambda model: False
    adapter.AdapterProcessor = type("AdapterProcessor", (), {})
    adapter.CrossAttentionAdapterMixin = type("CrossAttentionAdapterMixin", (), {})
    sys.modules[adapter.__name__] = adapter
    _load("detikzify.util.torch", ref / "util/torch.py")
    util.infer_device = sys.modules["detikzify.util.torch"].infer_device

    class Metric(torch.nn.Module):
        def __init__(self, **kwargs):
            super().__init__()
            self._defaults, self._dtype = {}, torch.float32

        def add_state(self, name, default, dist_reduce_fx=None):
            self._defaults[name] = default
            setattr(self, name, default.clone())

        def reset(self):
            for k, v in self._defaults.items():
                setattr(self, k, v.clone())

        def set_dtype(self, dtype):
            self._dtype = dtype
            return self

        device = property(lambda self: self._device)
        dtype = property(lambda self: self._dtype)
    tm.Metric = Metric
    tmf = types.ModuleType("torchmetrics.functional")
    tmf.pairwise_cosine_similarity = lambda a, b: torch.nn.functional.normalize(a, dim=-1) @ torch.nn.functional.normalize(b, dim=-1).T
    sys.modules["torchmetrics.functional"] = tmf
    ot, otlp = types.ModuleType("ot"), types.ModuleType("ot.lp")

    def emd2(M, a, b):   # POT's ot.lp.emd2 restated: the transport LP, empty marginals = uniform
        from scipy.optimize import linprog
        M = np.asarray(M, dtype=np.float64)
        n, m = M.shape
        a = np.full(n, 1.0 / n) if len(a) == 0 else np.asarray(a, dtype=np.float64)
        b = np.full(m, 1.0 / m) if len(b) == 0 else np.asarray(b, dtype=np.float64)
        A_eq = np.zeros((n + m, n * m))
        for i in range(n):
            A_eq[i, i * m:(i + 1) * m] = 1.0
        for j in range(m):
            A_eq[n + j, j::m] = 1.0
        res = linprog(M.reshape(-1), A_eq=A_eq, b_eq=np.concatenate([a, b]), bounds=(0, None), method="highs")
        assert res.status == 0, res.message
        return float(res.fun)
    otlp.emd2 = emd2
    sys.modules["ot"], sys.modules["ot.lp"] = ot, otlp
    _load("detikzify.evaluate.imagesim", ref / "evaluate/imagesim.py")
    tikz = types.ModuleType("detikzify.infer.tikz")

    class TikzDocument:
        """Stand-in for the TeX toolchain: every program 'compiles'."""
        def __init__(self, code, timeout=None):
            self.code, self.timeout = code, timeout
        is_rasterizable = True
        compiled_with_errors = False
        errors = {}

        def rasterize(self):
            return Image.new("RGB", (32, 32), "white")
    tikz.TikzDocument = TikzDocument
    sys.modules[tikz.__name__] = tikz
    return _load("detikzify.infer.generate", ref / "infer/generate.py")


def load_reference_image_processor(ref: Path):
    timm = types.ModuleType("timm")
    timm.__path__ = []
    data, models = types.ModuleType("timm.data"), types.ModuleType("timm.models")
    cfg = {"input_size": [3, 384, 384], "mean": (0.5, 0.5, 0.5), "std": (0.5, 0.5, 0.5), "crop_mode": "center"}
    models.resolve_pretrained_cfg = lambda variant: types.SimpleNamespace(to_dict=lambda: dict(cfg))
    data.resolve_data_config = lambda d: dict(d)
    sys.modules.update({"timm": timm, "timm.data": data, "timm.models": models})
    mod = _load("ref_processing_detikzify", ref / "model/v1/processing_detikzify.py")
    return mod.DetikzifyImageProcessor.from_pretrained("vit_so400m_patch14_siglip_384.webli")


def main(ref: Path):
    gen = load_reference_infer(ref)
    out, arrays = {}, {}

    model, proc, eng = _ours(eos_at=30)
    pipe = gen.DetikzifyPipeline(model=model, processor=proc, metric="fast")
    doc = pipe.sample(image=_figure())
    out["sample"] = {"gen_kwargs": {k: v for k, v in pipe.gen_kwargs.items() if isinstance(v, (bool, int, float, str))},
                     "doc": doc_json(doc), "sampling": sampling_json(eng.last_sampling), "calls": calls_json(eng.calls)}

    model, proc, eng = _ours(eos_at=36)
    pipe = gen.DetikzifyPipeline(model=model, processor=proc, metric="fast")
    results = list(pipe.simulate(image=_figure(), expansions=4))
    out["simulate_fast"] = {"scores": [float(s) for s, _ in results], "first_doc": doc_json(results[0][1])}

    model, proc, eng = _ours(eos_at=60)
    g = gen.DetikzifyGenerator(model=model, processor=proc, image=_figure(), metric=None, max_length=proc.tokenizer.model_max_length,
                               temperature=0.8, top_p=0.95, top_k=0, do_sample=True)
    res = [next(g.simulate(expansions=1)) for _ in range(2)]
    root = g.montecarlo.root_node
    out["generator_tree"] = {"scores": [float(s) for s, _ in res], "first_doc": doc_json(res[0][1]), "root_visits": root.visits,
                             "first_child_widen": root.children[0].is_widen_node,
                             "newlineinfo": {str(k): [v.num_lines, v.trailing] for k, v in sorted(g.newlineinfo.items())}}

    model, proc, eng = _ours(eos_at=36)
    pipe = gen.DetikzifyPipeline(model=model, processor=proc, metric="model")
    pipe.metric.update(img1=_figure(), img2=_figure())
    same = float(pipe.metric.compute())
    pipe.metric.reset()
    results = list(pipe.simulate(image=_figure(), expansions=3))
    out["simulate_selfsim"] = {"metric": str(pipe.metric), "mode": pipe.metric.mode, "same_figure": same,
                               "scores": [float(s) for s, _ in results], "first_doc": doc_json(results[0][1])}

    model, proc, eng = _ours(eos_at=36)
    sim = sys.modules["detikzify.evaluate.imagesim"].ImageSim.from_detikzify(model, proc, mode="emd")
    arrays["emd_f1"] = sim.get_vision_features(_figure()).double().numpy()
    arrays["emd_f2"] = sim.get_vision_features(_other()).double().numpy()
    out["emd"] = {"similarity": float(sim.get_similarity(_figure(), _other())), "same_figure": float(sim.get_similarity(_figure(), _figure()))}

    node = sys.modules["detikzify.mcts.node"].Node
    root, child = node("s"), node("c")
    root.add_child(child)
    child.update_policy_value(1.0)
    child.update_win_value(0.5)
    out["mcts_node"] = {"visits": root.visits, "win_value": root.win_value, "child_score": child.get_score(root),
                        "attributes": sorted(vars(root))}

    ip = load_reference_image_processor(ref)
    out["image_processor"] = {"size": ip.size, "image_mean": list(ip.image_mean), "image_std": list(ip.image_std),
                              "resample": int(ip.resample), "rescale_factor": ip.rescale_factor}
    for i, im in enumerate(_preprocess_inputs()):
        pv = ip(images=im, return_tensors="pt")["pixel_values"].double().numpy()
        # the normalised pixels are (k / 255 - 0.5) / 0.5 of 8-bit values k: stored as k, exact to far below the test's 1e-6
        k = np.rint((pv + 1.0) * 127.5)
        assert k.min() >= 0 and k.max() <= 255 and np.abs((k / 255 - 0.5) / 0.5 - pv).max() < 1e-7
        arrays[f"pixels_{i}"] = k.astype(np.uint8)

    (HERE / "reference_dropin.json").write_text(json.dumps(out, indent=1, sort_keys=True) + "\n")
    np.savez_compressed(HERE / "reference_dropin.npz", **arrays)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(Path(sys.argv[1]) / "detikzify")
