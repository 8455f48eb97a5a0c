"""Record, as data, what tests/test_dropin_cpu.py compares this project against in the original project's tree, so that the comparison
runs without that tree:  python tests/golden/make_reference_surface.py   (reads the tree named by _ref_import.REF)

Writes tests/golden/reference_surface.json:
  extract_box     outputs of the original `extract_box` (eval_img2text_seed_x_i.py) on fixed strings
  entry_scripts   per entry script eval_*.py: whether it builds the edit adapter, every `<name>.<attr>(...)` call with its keyword names,
                  and its import block (the top-level imports and the `setup_root` call) as structured records
  configs         the parsed inference YAMLs
  goldens         digests of every tensor make_golden.py writes when run against the original modules (tests/golden/*.pt)
  anyres          digests of the original any-res pre-processing on the seeded image sizes the test draws
No source code is stored: only names, keyword lists, parsed configs, strings and digests.
"""
import ast
import glob
import hashlib
import json
import os
import re
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(HERE, "reference_surface.json")

CONFIGS = ["visual_encoder/qwen_vitg_448.yaml", "processer/qwen_448_transform.yaml", "discrete_model/discrete_identity.yaml",
           "tokenizer/clm_llama_tokenizer_224loc_anyres.yaml", "clm_models/llm_seed_x.yaml", "clm_models/llm_seed_x_i.yaml",
           "clm_models/llm_seed_x_edit.yaml", "clm_models/llm_seed_x_lora.yaml", "clm_models/agent_seed_x.yaml", "clm_models/agent_seed_x_i.yaml",
           "clm_models/agent_seed_x_edit.yaml", "sdxl_adapter/sdxl_qwen_vit_resampler_l4_q64_pretrain_no_normalize.yaml",
           "sdxl_adapter/sdxl_qwen_vit_resampler_l4_q64_full_with_latent_image_pretrain_no_normalize.yaml"]
EXTRACT_BOX_INPUTS = ["The mask <box_start><loc-112><loc-56><loc-40><loc-20><box_end> and <box_start><loc-0><loc-223><loc-10><loc-5><box_end>.",
                      "none", "<box_start><loc-7><box_end><box_start><box_end>", "<box_start>a<loc-1>b<loc-22>c<box_end>"]
ANYRES_BASE = 448
ANYRES_GRIDS = ["1x1", "1x2", "1x3", "2x1", "3x1", "1x4", "4x1", "2x2"]
ANYRES_CASES = 60


def tensor_digest(t):
    """dtype, shape and SHA-256 of the contiguous bytes: equal digests <=> bit-identical tensors"""
    import torch
    t = t.detach().cpu().contiguous()
    return f"{t.dtype}:{list(t.shape)}:{hashlib.sha256(t.view(-1).view(torch.uint8).numpy().tobytes()).hexdigest()}"


def nested_digests(obj, path="", acc=None):
    """{path: digest} over a torch.load()ed golden: tensors by tensor_digest, every other leaf by repr"""
    import torch
    acc = {} if acc is None else acc
    if torch.is_tensor(obj):
        acc[path] = tensor_digest(obj)
    elif isinstance(obj, dict):
        for k in obj:
            nested_digests(obj[k], f"{path}/{k}", acc)
    elif isinstance(obj, (list, tuple)):
        acc[path + "#len"] = repr(len(obj))
        for i, x in enumerate(obj):
            nested_digests(x, f"{path}[{i}]", acc)
    else:
        acc[path] = repr(obj)
    return acc


def anyres_cases():
    """the seeded (image, grid list, keep-ratio check) cases of test_anyres_preprocessing_equals_the_reference_on_random_sizes"""
    import numpy as np
    from PIL import Image
    grids = [[ANYRES_BASE * int(g[0]), ANYRES_BASE * int(g[2])] for g in ANYRES_GRIDS]
    rng = np.random.RandomState(7)
    for i in range(ANYRES_CASES):
        w, h = int(rng.randint(40, 2600)), int(rng.randint(40, 2600))
        img = Image.fromarray(rng.randint(0, 255, (h, w, 3), dtype=np.uint8))
        yield i, w, h, img, (grids if i % 3 else grids[:1]), i % 10 == 0


def _call_record(node):
    f = node.func
    owner = f.value.id if isinstance(f.value, ast.Name) else None
    return {"owner": owner, "attr": f.attr, "args": [ast.literal_eval(a) if not isinstance(a, ast.Name) else {"name": a.id} for a in node.args],
            "kwargs": {k.arg: ast.literal_eval(k.value) for k in node.keywords}}


def entry_script_record(path):
    src = open(path).read()
    tree = ast.parse(src)
    calls = []
    for node in ast.walk(tree):
        if isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute) and isinstance(node.func.value, ast.Name):
            calls.append({"line": node.lineno, "owner": node.func.value.id, "attr": node.func.attr,
                          "keywords": sorted(k.arg for k in node.keywords if k.arg is not None)})
    block = []
    for node in tree.body:
        if isinstance(node, ast.Import):
            block.append({"import": [[a.name, a.asname] for a in node.names]})
        elif isinstance(node, ast.ImportFrom):
            block.append({"from": node.module, "level": node.level, "names": [[a.name, a.asname] for a in node.names]})
        elif isinstance(node, ast.Expr) and isinstance(node.value, ast.Call) and getattr(node.value.func, "attr", "") == "setup_root":
            block.append({"call": _call_record(node.value)})
    return {"edit": "with_latent_image" in src, "calls": calls, "import_block": block}


def main():
    import torch
    import yaml
    sys.path.insert(0, ROOT)
    sys.path.insert(0, HERE)
    import _ref_import
    ref = _ref_import.REF
    rec = {}

    ns = {}
    tree = ast.parse(open(os.path.join(ref, "src/inference/eval_img2text_seed_x_i.py")).read())
    fn = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "extract_box")
    exec(compile(ast.Module(body=[fn], type_ignores=[]), "extract_box", "exec"), {"re": re}, ns)
    rec["extract_box"] = [[s, ns["extract_box"](s)] for s in EXTRACT_BOX_INPUTS]

    scripts = sorted(glob.glob(os.path.join(ref, "src/inference/eval_*.py")))
    rec["entry_scripts"] = {os.path.basename(p): entry_script_record(p) for p in scripts}
    rec["configs"] = {n: yaml.safe_load(open(os.path.join(ref, "configs", n))) for n in CONFIGS}

    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([sys.executable, os.path.join(HERE, "make_golden.py")], cwd=ROOT, env=dict(os.environ, SEEDX_GOLDEN_OUT=d),
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-3000:]
        rec["goldens"] = {f: nested_digests(torch.load(os.path.join(d, f))) for f in sorted(os.listdir(d)) if f.endswith(".pt")}

    ar, tr = _ref_import.ref_module("src.inference.any_res"), _ref_import.ref_module("src.processer.transforms")
    cases = []
    for i, w, h, img, grids, keep in anyres_cases():
        views, pos = ar.process_anyres_image(img, tr.get_transform("clip", keep_ratio=False, image_size=ANYRES_BASE), grids, ANYRES_BASE)
        c = {"i": i, "w": w, "h": h, "views": tensor_digest(views), "patch_positions": tensor_digest(pos)}
        if keep:
            c["keep_ratio"] = tensor_digest(tr.get_transform("clip", keep_ratio=True, image_size=ANYRES_BASE)(img))
        cases.append(c)
    rec["anyres"] = cases

    with open(OUT, "w") as f:
        json.dump(rec, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
