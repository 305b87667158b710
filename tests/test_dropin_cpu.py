"""CPU: INTEGRATION.md §1 — with LLAVA_REFERENCE_ROOT set, the reference's OWN consumers of the hot path (llava/serve/cli.py,
llava/serve/model_worker.py, llava/eval/model_vqa_loader.py, llava/eval/run_llava.py) import on top of this package's
`llava.model`, and the entry points they call have the reference's signatures. What the reference's files import, its
signatures and its stopping criterion's verdicts are recorded in tests/golden/reference_interface.json
(tests/golden/make_reference_interface.py), so these tests need no reference tree."""
import inspect
import json
import os
import subprocess
import sys
import textwrap

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_interface.json")


def _golden():
    with open(GOLD) as f:
        return json.load(f)


def _write_reference_stand_in(root, g):
    """A reference tree whose modules carry the reference's own module-level `from llava... import` statements; the names
    other modules import from a stand-in are defined in it as placeholders."""
    exported = {}
    for imps in g["imports"].values():
        for src, names in imps:
            exported.setdefault(src, set()).update(names)
    for pkg in g["packages"]:
        os.makedirs(os.path.join(root, *pkg.split(".")), exist_ok=True)
        open(os.path.join(root, *pkg.split("."), "__init__.py"), "w").close()
    for mod, imps in g["imports"].items():
        path = os.path.join(root, *mod.split(".")) + ".py"
        os.makedirs(os.path.dirname(path), exist_ok=True)
        lines = [f"from {src} import {', '.join(names)}" for src, names in imps]
        imported = {n for _, names in imps for n in names}
        lines += [f"{n} = None" for n in sorted(exported.get(mod, set()) - imported)]
        with open(path, "w") as f:
            f.write("\n".join(lines) + "\n")


def test_reference_consumers_import_on_top_of_this_package(repo_root, tmp_path):
    g = _golden()
    ref = str(tmp_path / "reference")
    _write_reference_stand_in(ref, g)
    code = textwrap.dedent("""
        import importlib, json, sys
        import llava
        pkg, ref, g = sys.argv[1], sys.argv[2], json.load(open(sys.argv[3]))
        import llava.model.builder as b, llava.model.language_model.llava_llama as ll, llava.model.llava_arch as arch
        import llava.constants as c
        for name in g["imports"]:
            m = importlib.import_module(name)
            assert m.__file__.startswith(ref), m.__file__          # the reference's files
        for m in (b, ll, arch, c):
            assert m.__file__.startswith(pkg), m.__file__          # the hot path: this repo
        for name in g["consumers"]:
            assert importlib.import_module(name).load_pretrained_model is b.load_pretrained_model, name
        for k, v in g["constants"].items():
            assert getattr(c, k) == v, (k, getattr(c, k), v)
        assert importlib.import_module("llava.mm_utils").IMAGE_TOKEN_INDEX == -200
        print("ok")
    """)
    pkg = os.path.join(repo_root, "llava-plus-codebase_b200")
    env = dict(os.environ, LLAVA_REFERENCE_ROOT=ref, PYTHONPATH=pkg, TRANSFORMERS_OFFLINE="1", HF_HUB_OFFLINE="1")
    r = subprocess.run([sys.executable, "-c", code, pkg, ref, GOLD], cwd=tmp_path, env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0 and "ok" in (r.stdout + r.stderr).splitlines()[-1], r.stderr[-2000:]


def test_entry_point_signatures_match_the_reference():
    from llava.model.builder import load_pretrained_model
    from llava.model.language_model.llava_llama import LlavaLlamaForCausalLM
    from llava.model.multimodal_encoder.builder import build_vision_tower
    from llava.model.multimodal_projector.builder import build_vision_projector

    ref = {s["func"]: s["params"] for s in _golden()["signatures"]}
    ours = list(inspect.signature(load_pretrained_model).parameters)
    assert ours[: len(ref["load_pretrained_model"])] == ref["load_pretrained_model"]
    assert list(inspect.signature(LlavaLlamaForCausalLM.forward).parameters) == ref["forward"]
    assert list(inspect.signature(LlavaLlamaForCausalLM.prepare_inputs_labels_for_multimodal).parameters) == \
        ref["prepare_inputs_labels_for_multimodal"]
    assert list(inspect.signature(LlavaLlamaForCausalLM.encode_images).parameters) == ref["encode_images"]
    assert list(inspect.signature(build_vision_tower).parameters)[0] == ref["build_vision_tower"][0]
    assert list(inspect.signature(build_vision_projector).parameters)[:2] == ref["build_vision_projector"][:2]


def test_reference_keywords_stopping_criteria_through_the_decode_loop():
    """The reference's OWN KeywordsStoppingCriteria (llava/mm_utils.py:79-114), replayed from its recorded verdict on every
    prefix of the generation, driving generate()'s host loop: the loop must hand it cat(prompt ids incl. IMAGE_TOKEN_INDEX,
    new tokens), one column more per step, and stop at the step whose tail spells the keyword (GPU counterpart with a
    restated criterion: tests/test_generate_gpu.py)."""
    import torch

    from llava.model.language_model.llava_llama import _stream_decode
    from test_generate_host import FakeEngine, per_step_reference

    k = _golden()["keywords_stopping"]
    free = per_step_reference([4], 40, set(), 0)[0].tolist()           # what the fake model generates unconstrained
    assert free == k["free_tokens"], "the fake model drifted from the recorded generation"
    stop_at = k["stop_at"]
    assert k["verdicts"].index(True) + 1 == stop_at and k["start_len"] == len(k["prompt"]) == 5

    class RecordedKeywordsCriterion:
        def __init__(self):
            self.calls = 0

        def __call__(self, output_ids, scores, **kw):
            self.calls += 1
            n = output_ids.shape[1] - k["start_len"]
            assert n == self.calls, (n, self.calls)
            assert output_ids.tolist() == [k["prompt"] + free[:n]]
            return k["verdicts"][n - 1]

    crit = RecordedKeywordsCriterion()
    out = _stream_decode(FakeEngine([4]), None, None, None, 1, 40, set(), 0, torch.tensor([k["prompt"]]), None, [crit],
                         run_ahead=8)
    assert out[0].tolist() == free[:stop_at] and crit.calls == stop_at
