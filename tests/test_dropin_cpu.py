"""Drop-in surface checked without a GPU: prompt layouts, grounding post-processing, the launcher for unmodified reference scripts, and
checks against the reference's own entry scripts, configs, goldens and pre-processing.  What those checks compare against was recorded
from the reference tree into tests/golden/reference_surface.json (tests/golden/make_reference_surface.py), so they run without it."""
import ast
import inspect
import json
import os
import subprocess
import sys

import pytest
import torch

from seedx_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, GOLDEN)
import make_reference_surface as surface  # noqa: E402

REF = json.load(open(os.path.join(GOLDEN, "reference_surface.json")))


def test_chat_prompt_layout_single_and_multi_turn():
    from seedx_b200 import demo
    tok = synth.SynthTokenizer()
    q = "What is in the image?"
    a_ids, a_mask = demo.image_prompt(tok, 3, q)
    b_ids, b_mask = demo.chat_prompt(tok, [q], views_per_image=[3])
    assert torch.equal(a_ids, b_ids) and torch.equal(a_mask, b_mask)          # one turn, one image == the eval_img2text layout
    assert int(a_mask.sum()) == 3 * 64
    # the layout of eval_img2text_seed_x_i.py:142-147 spelled out
    img = "".join("<img_{:05d}>".format(i) for i in range(64))
    text = "[INST] " + ("<patch>" + img + "</patch>") * 2 + "<img>" + img + "</img>" + q + " [/INST]\n"
    assert a_ids[0].tolist() == [tok.bos_token_id] + tok.encode(text)
    # two images (2 + 1 views), three turns, system message
    ids, mask = demo.chat_prompt(tok, ["q1", "a1", "q2"], views_per_image=[2, 1], system_message="sys")
    assert int(mask.sum()) == 3 * 64
    want = "sys\n[INST] " + "<patch>" + img + "</patch>" + "<img>" + img + "</img>" + "<img>" + img + "</img>" + "q1 [/INST]\na1\n[INST] q2 [/INST]\n"
    assert ids[0].tolist() == [tok.bos_token_id] + tok.encode(want)
    # masked rows are exactly the <img_k> ids, in order, once per view
    first = tok.tok2id["<img_00000>"]
    assert ids[0][mask[0]].tolist() == list(range(first, first + 64)) * 3
    ids_f, _ = demo.chat_prompt(tok, ["draw a cat"], force_image=True)
    assert ids_f[0, -1].item() == tok.tok2id["<img>"]
    with pytest.raises(ValueError):
        demo.chat_prompt(tok, ["q1", "a1"])


def test_extract_box_and_pixel_corners():
    from seedx_b200 import demo
    s = "The mask <box_start><loc-112><loc-56><loc-40><loc-20><box_end> and <box_start><loc-0><loc-223><loc-10><loc-5><box_end>."
    assert demo.extract_box(s) == [[112, 56, 40, 20], [0, 223, 10, 5]]
    assert demo.extract_box("no boxes here <loc-3>") is None
    # (x_center, y_center, w, h) in 224 bins on a 448 x 896 image
    assert demo.box_to_pixels([112, 56, 40, 20], 448, 896) == (184, 184, 264, 264)
    assert demo.box_to_pixels([0, 223, 10, 5], 448, 896) == (-10, 882, 10, 902)
    # the reference's own extract_box (eval_img2text_seed_x_i.py) on the same strings
    assert [t for t, _ in REF["extract_box"]] == [s, "none", "<box_start><loc-7><box_end><box_start><box_end>", "<box_start>a<loc-1>b<loc-22>c<box_end>"]
    for t, want in REF["extract_box"]:
        assert demo.extract_box(t) == want, t


def test_visualize_bbox_draws_the_rectangle(tmp_path):
    import numpy as np
    from PIL import Image
    from seedx_b200 import demo
    img = Image.new("RGB", (448, 224), (0, 0, 0))
    out = demo.visualize_bbox(img, [[112, 112, 56, 56]], str(tmp_path / "vis" / "g.png"))
    a = np.asarray(out)
    x1, y1, x2, y2 = demo.box_to_pixels([112, 112, 56, 56], 448, 224)
    assert (x1, y1, x2, y2) == (168, 84, 280, 140)
    assert tuple(a[y1, x1]) == (0, 255, 0) and tuple(a[y2, x2]) == (0, 255, 0) and tuple(a[(y1 + y2) // 2, (x1 + x2) // 2]) == (0, 0, 0)
    assert os.path.exists(tmp_path / "vis" / "g.png")


def test_launcher_runs_a_reference_style_script(tmp_path):
    """a script that begins like the reference's (top-level third-party imports, pyrootutils marker, sibling import, YAML `_target_`)
    runs unmodified through `python -m seedx_b200.run` even though hydra / omegaconf / pyrootutils / diffusers are not installed"""
    d = tmp_path / "proj" / "src" / "inference"
    os.makedirs(d)
    open(tmp_path / "proj" / ".project-root", "w").close()
    (d / "any_res.py").write_text("def process_anyres_image(*a):\n    return 'sibling import ok'\n")
    (d / "eval_demo.py").write_text(
        "import hydra\nimport torch\nimport os\nimport pyrootutils\nfrom omegaconf import OmegaConf\n"
        "from diffusers import AutoencoderKL, UNet2DConditionModel, EulerDiscreteScheduler\n"
        "from any_res import process_anyres_image\n"
        "root = pyrootutils.setup_root(__file__, indicator='.project-root', pythonpath=True)\n"
        "import sys\nassert __name__ == '__main__' and sys.argv[1:] == ['--flag']\n"
        "cfg = OmegaConf.load('configs/processer/qwen_448_transform.yaml')\n"
        "t = hydra.utils.instantiate(cfg)\n"
        "lc = OmegaConf.load('configs/clm_models/llm_seed_x_lora.yaml')\n"
        "print('OK', callable(t), process_anyres_image(), os.path.basename(str(root)), lc.peft_config.r, lc['vocab_size'])\n")
    r = subprocess.run([sys.executable, "-m", "seedx_b200.run", str(d / "eval_demo.py"), "--flag"], cwd=ROOT, capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip().endswith("OK True sibling import ok proj 32 32330"), r.stdout


# ---- checks against the reference's own entry scripts, configs, goldens and pre-processing (recorded in tests/golden/reference_surface.json) --
def _named_params(fn):
    return {p.name for p in inspect.signature(fn).parameters.values() if p.kind in (p.POSITIONAL_OR_KEYWORD, p.KEYWORD_ONLY)}


def test_reference_scripts_only_use_keywords_the_replacement_names():
    from seedx_b200 import compat
    compat.install()
    from seedx_b200.adapter import SDXLAdapter, SDXLAdapterWithLatentImage
    from seedx_b200.agent import ContinuousLVLM
    from seedx_b200.sdxl import AutoencoderKL, EulerDiscreteScheduler, UNet2DConditionModel
    scripts = REF["entry_scripts"]
    assert len(scripts) == 7
    seen = 0
    for name, script in sorted(scripts.items()):
        adapter_cls = SDXLAdapterWithLatentImage if script["edit"] else SDXLAdapter
        for c in script["calls"]:
            kws, owner = set(c["keywords"]), c["owner"]
            if c["attr"] == "generate" and owner == "agent_model":
                target = ContinuousLVLM.generate
            elif c["attr"] == "generate" and owner == "adapter":
                target = adapter_cls.generate
            elif c["attr"] == "init_pipe" and owner == "adapter":
                target = adapter_cls.init_pipe
            elif c["attr"] == "from_pretrained" and owner in ("AutoencoderKL", "UNet2DConditionModel", "EulerDiscreteScheduler"):
                target = {"AutoencoderKL": AutoencoderKL, "UNet2DConditionModel": UNet2DConditionModel,
                          "EulerDiscreteScheduler": EulerDiscreteScheduler}[owner].from_pretrained
            else:
                continue
            missing = kws - _named_params(target)
            assert not missing, f"{name}:{c['line']} passes {sorted(missing)} which {target.__qualname__} does not name"
            seen += 1
    assert seen >= 20, seen


def _import_block_module(block):
    """the recorded import block of one entry script as a module: its imports and its `setup_root(...)` statement, in order"""
    body = []
    for st in block:
        if "import" in st:
            body.append(ast.Import(names=[ast.alias(name=n, asname=a) for n, a in st["import"]]))
        elif "from" in st:
            body.append(ast.ImportFrom(module=st["from"], names=[ast.alias(name=n, asname=a) for n, a in st["names"]], level=st["level"]))
        else:
            c = st["call"]
            args = [ast.Name(id=a["name"], ctx=ast.Load()) if isinstance(a, dict) else ast.Constant(a) for a in c["args"]]
            func = ast.Attribute(value=ast.Name(id=c["owner"], ctx=ast.Load()), attr=c["attr"], ctx=ast.Load())
            body.append(ast.Expr(ast.Call(func=func, args=args, keywords=[ast.keyword(arg=k, value=ast.Constant(v)) for k, v in c["kwargs"].items()])))
    return ast.fix_missing_locations(ast.Module(body=body, type_ignores=[]))


def test_import_block_of_every_reference_entry_script_executes_under_the_stand_ins():
    """the statements every reference entry script runs before touching a model — its top-level imports (incl. `from diffusers import …,
    Transformer2DModel` and the sibling `from any_res import …`) and `pyrootutils.setup_root` — execute against this repo exactly as
    `python -m seedx_b200.run <script>` would run them (compat.install() + script directory on sys.path); a missing name fails here, not on a GPU box"""
    scripts = REF["entry_scripts"]
    assert len(scripts) == 7
    blocks = {name: ast.unparse(_import_block_module(s["import_block"])) for name, s in sorted(scripts.items())}
    for name, s in scripts.items():
        assert len(s["import_block"]) >= 7, name
        assert s["import_block"][-1]["call"]["attr"] == "setup_root", name
    code = r'''
import os, sys
sys.path.insert(0, %r)
from seedx_b200 import compat
compat.install()
sys.path.insert(0, os.path.join(%r, "src", "inference"))      # what seedx_b200.run does for the sibling import
for name, block in %r.items():
    # __file__ of the script as the launcher sees it: the same relative location inside THIS repo
    ns = {"__name__": "not_main", "__file__": os.path.join(%r, "src", "inference", name)}
    exec(compile(block, name, "exec"), ns)
    import diffusers
    for n in ("AutoencoderKL", "UNet2DConditionModel", "EulerDiscreteScheduler"):
        assert ns[n] is getattr(diffusers, n)
    print("ok", name)
''' % (ROOT, ROOT, blocks, ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    assert r.stdout.count("ok eval_") == 7, r.stdout


def test_reference_yaml_targets_resolve_with_identical_keys():
    """every inference YAML of the reference has a twin here with the same `_target_`s and keys (values may differ only in comments)"""
    import yaml
    from seedx_b200 import compat
    names = ["visual_encoder/qwen_vitg_448.yaml", "processer/qwen_448_transform.yaml", "discrete_model/discrete_identity.yaml",
             "tokenizer/clm_llama_tokenizer_224loc_anyres.yaml", "clm_models/llm_seed_x.yaml", "clm_models/llm_seed_x_i.yaml",
             "clm_models/llm_seed_x_edit.yaml", "clm_models/llm_seed_x_lora.yaml", "clm_models/agent_seed_x.yaml", "clm_models/agent_seed_x_i.yaml",
             "clm_models/agent_seed_x_edit.yaml", "sdxl_adapter/sdxl_qwen_vit_resampler_l4_q64_pretrain_no_normalize.yaml",
             "sdxl_adapter/sdxl_qwen_vit_resampler_l4_q64_full_with_latent_image_pretrain_no_normalize.yaml"]
    assert sorted(REF["configs"]) == sorted(names)

    def targets(o, acc):
        if isinstance(o, dict):
            if "_target_" in o:
                acc.append(o["_target_"])
            for v in o.values():
                targets(v, acc)
        return acc

    for n in names:
        ours = yaml.safe_load(open(os.path.join(ROOT, "configs", n)))
        ref = REF["configs"][n]
        assert ours == ref, n
        for t in targets(ours, []):
            if t.startswith(("src.", "peft.")):
                compat.install()
                assert callable(compat._locate(t)), t


def test_goldens_regenerate_bit_identically_from_the_reference():
    """tests/golden/*.pt ARE the outputs of the reference's own modules: every committed tensor is bit-identical (dtype, shape, SHA-256 of
    its bytes) and every other value equal to what tests/golden/make_golden.py wrote when it was run against the reference modules"""
    names = sorted(f for f in os.listdir(GOLDEN) if f.endswith(".pt"))
    assert names == sorted(REF["goldens"]) and len(names) == 8
    for f in names:
        got, want = surface.nested_digests(torch.load(os.path.join(GOLDEN, f))), REF["goldens"][f]
        assert got.keys() == want.keys(), f
        for k in want:
            assert got[k] == want[k], f"{f}{k}"


def test_anyres_preprocessing_equals_the_reference_on_random_sizes():
    """seedx_b200.preprocess vs the reference's own functions: grid choice, tile order, patch positions and pixel values, bit for bit
    (dtype, shape and SHA-256 of the reference's outputs), on 60 random image sizes and both transform modes"""
    from seedx_b200 import preprocess as pp
    base = surface.ANYRES_BASE
    cases = REF["anyres"]
    assert len(cases) == 60
    n = 0
    for (i, w, h, img, grids, keep), want in zip(surface.anyres_cases(), cases):
        assert (i, w, h) == (want["i"], want["w"], want["h"])
        v1, p1 = pp.process_anyres_image(img, pp.get_transform("clip", keep_ratio=False, image_size=base), grids, base)
        assert surface.tensor_digest(v1) == want["views"] and surface.tensor_digest(p1) == want["patch_positions"], (w, h)
        assert keep == ("keep_ratio" in want)
        if keep:
            k1 = pp.get_transform("clip", keep_ratio=True, image_size=base)(img)
            assert surface.tensor_digest(k1) == want["keep_ratio"], (w, h)
        n += 1
    assert n == 60
