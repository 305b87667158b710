"""What tests/test_dropin_cpu.py compares against, recorded from the unmodified reference into reference_interface.json:

- the `from llava.<module> import <names>` statements at module level of the reference's own consumers of the hot path
  (llava/serve/cli.py, llava/serve/model_worker.py, llava/eval/model_vqa_loader.py, llava/eval/run_llava.py) and of the
  reference modules they pull in, and the reference's values of the llava.constants names among them;
- the parameter lists of the hot-path entry points (load_pretrained_model, forward, prepare_inputs_labels_for_multimodal,
  encode_images, build_vision_tower, build_vision_projector);
- the verdict of the reference's KeywordsStoppingCriteria (llava/mm_utils.py) on every prefix of one generation.

    python tests/golden/make_reference_interface.py     (needs the reference tree, LLAVA_REFERENCE_ROOT)
"""
import ast
import json
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "llava-plus-codebase_b200"), os.path.join(ROOT, "tests")]
from oracle.ref_shim import REFERENCE_ROOT  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_interface.json")
CONSUMERS = ["llava.serve.cli", "llava.serve.model_worker", "llava.eval.model_vqa_loader", "llava.eval.run_llava"]
HOT_PATH = ("llava.constants", "llava.model")   # what this package implements; every other llava module is the reference's
SIGNATURES = [("model/builder.py", None, "load_pretrained_model"),
              ("model/language_model/llava_llama.py", "LlavaLlamaForCausalLM", "forward"),
              ("model/llava_arch.py", "LlavaMetaForCausalLM", "prepare_inputs_labels_for_multimodal"),
              ("model/llava_arch.py", "LlavaMetaForCausalLM", "encode_images"),
              ("model/multimodal_encoder/builder.py", None, "build_vision_tower"),
              ("model/multimodal_projector/builder.py", None, "build_vision_projector")]
PROMPT = [1, 5, -200, 7, 9]


def _path(module):
    base = os.path.join(REFERENCE_ROOT, *module.split("."))
    return base + ".py" if os.path.exists(base + ".py") else os.path.join(base, "__init__.py")


def _imports(module):
    """[[from-module, [names]], ...] of the module-level `from llava... import` statements, in file order."""
    tree = ast.parse(open(_path(module)).read())
    out = []
    for node in tree.body:
        if isinstance(node, ast.ImportFrom) and node.level == 0 and (node.module or "").split(".")[0] == "llava":
            out.append([node.module, [a.name for a in node.names]])
        elif isinstance(node, ast.Import):
            assert not any(a.name.split(".")[0] == "llava" for a in node.names), (module, "plain `import llava...`")
    return out


def consumer_imports():
    mods, todo = {}, list(CONSUMERS)
    while todo:
        m = todo.pop(0)
        if m in mods:
            continue
        mods[m] = _imports(m)
        todo += [src for src, _ in mods[m] if not src.startswith(HOT_PATH)]
    return mods


def signature(rel, cls, func):
    tree = ast.parse(open(os.path.join(REFERENCE_ROOT, "llava", rel)).read())
    scope = tree.body if cls is None else next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == cls).body
    fn = next(n for n in scope if isinstance(n, ast.FunctionDef) and n.name == func)
    return [a.arg for a in fn.args.args]


class Tok:
    """Letters a..z for ids 0..25 (mod 26), bos = 1: enough of a tokenizer for KeywordsStoppingCriteria."""
    bos_token_id = 1

    def __call__(self, text):
        return type("Enc", (), {"input_ids": [1] + [ord(c) - 97 for c in text]})()

    def batch_decode(self, ids, skip_special_tokens=True):
        return ["".join(chr(97 + int(i) % 26) if int(i) >= 0 else "?" for i in row) for row in ids]


def keyword_verdicts():
    import torch

    from test_generate_host import per_step_reference

    pkg = types.ModuleType("llava")
    pkg.__path__ = [os.path.join(REFERENCE_ROOT, "llava")]
    sys.modules["llava"] = pkg
    import llava.mm_utils as mu  # the reference's own file

    free = per_step_reference([4], 40, set(), 0)[0].tolist()
    text = "".join(chr(97 + t % 26) for t in free)
    keyword = text[6:9]
    prompt = torch.tensor([PROMPT])
    crit = mu.KeywordsStoppingCriteria([keyword], Tok(), prompt)
    verdicts = [bool(crit(torch.cat([prompt, torch.tensor([free[:k]])], 1), None)) for k in range(1, len(free) + 1)]
    return dict(prompt=PROMPT, free_tokens=free, keyword=keyword, start_len=int(crit.start_len),
                stop_at=text.find(keyword) + 3, verdicts=verdicts)


def main():
    mods = consumer_imports()
    const = sorted({n for imps in mods.values() for src, names in imps if src == "llava.constants" for n in names})
    ref_const = {}
    exec(open(_path("llava.constants")).read(), ref_const)
    out = dict(consumers=CONSUMERS, hot_path=list(HOT_PATH), imports=mods,
               constants={n: ref_const[n] for n in const},
               packages=sorted(m for m in {m.rsplit(".", 1)[0] for m in mods} if os.path.exists(_path(m))),
               signatures=[dict(file=rel, cls=cls, func=func, params=signature(rel, cls, func)) for rel, cls, func in SIGNATURES],
               keywords_stopping=keyword_verdicts())
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("wrote", os.path.basename(OUT))


if __name__ == "__main__":
    assert os.path.isdir(os.path.join(REFERENCE_ROOT, "llava", "serve")), "reference tree not found (set LLAVA_REFERENCE_ROOT)"
    main()
