"""Host-side logic and the closed-form approximations the kernels use, checked on the CPU (no GPU, no compute calls into the library)."""
import json
import math
import os
import subprocess
import sys

import pytest
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_exp2_polynomial_of_the_attention_kernels():
    """attention_pp.cu / attention_tc.cu `exp2_poly3`: x = n + f, 2^f by a degree-3 minimax polynomial, 2^n through the exponent field.
    Restated in numpy float32 with the same operation order; relative error must stay below the fp16 rounding of P (4.9e-4)."""
    src = open(os.path.join(ROOT, "seed-x_b200", "csrc", "attention_pp.cu")).read()
    for c in ("0.0551716685f", "0.2426111251f", "0.6932609677f", "0.9999280572f", "12582912.0f"):
        assert c in src, "coefficient %s changed in the kernel: update this restatement" % c
    x = np.linspace(-30.0, 8.5, 200001).astype(np.float32)
    t = (x + np.float32(12582912.0)).astype(np.float32)
    f = (x - (t - np.float32(12582912.0))).astype(np.float32)
    q = np.float32(0.0551716685) * f + np.float32(0.2426111251)
    q = q * f + np.float32(0.6932609677)
    q = q * f + np.float32(0.9999280572)
    r = (q.view(np.int32) + (t.view(np.int32) << 23)).view(np.float32)
    ref = np.exp2(x.astype(np.float64))
    assert np.abs(r / ref - 1).max() < 1.0e-4
    assert np.abs(f).max() <= 0.5 + 1e-6


def test_gelu_and_silu_closed_forms_of_the_gemm_epilogue():
    """common.cuh `gelu_erf_fast` (Abramowitz-Stegun 7.1.26 in FMA form) and `silu` vs torch, fp32."""
    x = torch.linspace(-12, 12, 100001, dtype=torch.float32)
    ax = x.abs()
    z = ax * 0.70710678118654752440
    t = 1.0 / (0.3275911 * z + 1.0)
    poly = t * 1.061405429 - 1.453152027
    poly = poly * t + 1.421413741
    poly = poly * t - 0.284496736
    poly = poly * t + 0.254829592
    poly = poly * t
    w = ax * 0.84932180028801904272
    erf_abs = 1.0 - poly * torch.exp2(-w * w)
    gelu = 0.5 * ax * erf_abs + 0.5 * x
    assert (gelu - torch.nn.functional.gelu(x.double()).float()).abs().max() < 5e-7 * 12
    silu = x / (1.0 + torch.exp2(-1.4426950408889634 * x))
    assert (silu - torch.nn.functional.silu(x.double()).float()).abs().max() < 1e-5


def test_static_condition_tree_helpers():
    from seedx_b200.sampler import _copy_tree, _same_layout
    a = dict(n_ctx=4, down=[[torch.zeros(2, 3)], [torch.zeros(5)]], aug=torch.zeros(2, 2))
    b = dict(n_ctx=4, down=[[torch.ones(2, 3)], [torch.full((5,), 2.0)]], aug=torch.full((2, 2), 3.0))
    assert _same_layout(a, b)
    ptr = a["down"][0][0].data_ptr()
    _copy_tree(a, b)
    assert a["down"][0][0].data_ptr() == ptr and float(a["down"][0][0].sum()) == 6.0 and float(a["aug"][0, 0]) == 3.0
    assert not _same_layout(a, dict(b, n_ctx=5))
    assert not _same_layout(a, dict(b, aug=torch.zeros(2, 3)))
    assert not _same_layout(a, dict(n_ctx=4, down=[[torch.ones(2, 3)]], aug=b["aug"]))


def test_launch_accounting_counts_graph_replays():
    from seedx_b200 import _lib
    n0 = _lib.launch_count()
    _lib.note_replay(960)
    _lib.note_replay(205)
    assert _lib.launch_count() - n0 == 1165


def test_groupnorm_workspace_size_covers_every_resolution():
    """seedx_groupnorm_ws_bytes(n, groups) must bound final stats + per-CTA partials + tickets for any hw (host arithmetic only)."""
    import ctypes as C
    from seedx_b200._lib import lib
    f = lib().seedx_groupnorm_ws_bytes
    for n in (1, 2, 8, 16, 64):
        got = f(C.c_int64(n), C.c_int(32))
        for hw in (64, 1024, 4096, 16384, 1 << 20):
            spb = max(32, -(-hw * n // 592))
            spb = min(spb, hw)
            nblk = -(-hw // spb)
            need = n * 32 * 2 * 8 + n * nblk * 32 * 2 * 4 + n * 4
            assert got >= need, (n, hw, got, need)


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["cpu_baseline"]["kind"] in ("port", "reference") and line["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0 and math.isfinite(line["value"])


def test_bench_output_dump_is_float32_exact_and_sampled_reproducibly_over_budget(tmp_path, monkeypatch):
    """bench.py --dump-outputs: uint8 pixels and token ids land exactly in float32; over the byte budget every array is cut to the same
    seeded sample of its elements on every run, in index order, and the files stay within the budget"""
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (2, 64, 64, 3), dtype=np.uint8)
    ids = [[7, 31000, 2], [5, 6, 32329]]
    bench.dump_outputs(str(tmp_path / "a"), {"images": img, "text_ids": ids})
    a_img, a_ids = np.load(tmp_path / "a" / "images.npy"), np.load(tmp_path / "a" / "text_ids.npy")
    assert a_img.dtype == np.float32 and np.array_equal(a_img, img) and np.array_equal(a_ids, np.array(ids))
    monkeypatch.setattr(bench, "DUMP_BYTES", 20000)
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), {"images": img, "text_ids": ids})
    b_img, c_img = np.load(tmp_path / "b" / "images.npy"), np.load(tmp_path / "c" / "images.npy")
    assert b_img.ndim == 1 and 0 < b_img.size < img.size and np.array_equal(b_img, c_img)
    assert sum(os.path.getsize(tmp_path / "b" / f) for f in os.listdir(tmp_path / "b")) <= 20000
    assert np.isin(b_img, img.reshape(-1)).all()


def test_reference_arm_under_torchrun_prints_once():
    """launched the way the driver launches N>1 (torch.distributed.run, one process per rank): rank 0 alone times and prints the line,
    the other ranks exit 0 without output"""
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                          "--master-port", str(port), os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["n_gpus"] == 2 and line["value"] > 0


def test_lora_merge_updates_the_packed_weights_in_place():
    """LlamaForCausalLM.apply_peft_state_dict on host tensors (no kernel is involved at load time): the packed [q|k|v] / [up,gate]-interleaved
    fp16 weights equal the fp16 rounding of W + (alpha/r) B A from seedx_b200.lora.merge_lora_state_dict, norms are replaced, storage
    pointers are unchanged (captured decode graphs stay valid), and the vocabulary growth follows peft_models.py:62-82."""
    import os
    import torch
    from seedx_b200 import lora, synth
    from seedx_b200._lib import SeedxError
    from seedx_b200.llm import LlamaForCausalLM
    g = torch.load(os.path.join(os.path.dirname(__file__), "golden", "llama_lora_tiny.pt"))
    cfg = dict(synth.TINY_LLAMA)
    base = synth.llama_state_dict(cfg)
    m = LlamaForCausalLM(cfg, max_len=64, device="cpu")
    m.load_state_dict({k: v.clone() for k, v in base.items()})        # on the host .to() may alias the caller's tensors
    m.resize_token_embeddings(g["new_vocab"])
    assert m.config.vocab_size == g["new_vocab"] and m.logits.shape[1] == g["new_vocab"]
    assert torch.allclose(m.embed[cfg["vocab"]:].float(), g["embed_new_rows"], atol=1e-3)
    assert torch.allclose(m.lm_head[cfg["vocab"]:].float(), g["head_new_rows"], atol=1e-3)
    ft = synth.lora_fixture(g["shapes"])
    with pytest.raises(SeedxError):
        m.apply_peft_state_dict(ft)                                     # no peft_config
    # the real peft.LoraConfig is a dataclass with r / lora_alpha and NO `.scaling` property (peft 0.4.0 config.py): a plain object stands for it
    import types
    m.peft_config = types.SimpleNamespace(r=g["r"], lora_alpha=g["lora_alpha"])
    ptrs = [L["wqkv"].data_ptr() for L in m.layers] + [L["wgu"].data_ptr() for L in m.layers]
    extra = m.apply_peft_state_dict({**ft, "base_model.model.model.layers.0.self_attn.rotary_emb.inv_freq": torch.zeros(4),
                                     "base_model.model.model.layers.9.mlp.up_proj.weight": torch.zeros(2, 2)})
    assert extra == ["model.layers.9.mlp.up_proj.weight"]               # reported like load_state_dict(strict=False)'s unexpected keys
    assert ptrs == [L["wqkv"].data_ptr() for L in m.layers] + [L["wgu"].data_ptr() for L in m.layers]
    full = {"base_model.model." + k: v for k, v in base.items()}
    full.update(ft)
    merged = lora.merge_lora_state_dict(full, g["lora_alpha"] / g["r"])
    D = cfg["hidden"]
    for i, L in enumerate(m.layers):
        p = f"model.layers.{i}."
        for j, n in enumerate(("q_proj", "k_proj", "v_proj")):
            assert torch.equal(L["wqkv"][j * D:(j + 1) * D], merged[p + f"self_attn.{n}.weight"].half())
        assert torch.equal(L["wo"], merged[p + "self_attn.o_proj.weight"].half())
        assert torch.equal(L["wgu"][0::2], merged[p + "mlp.up_proj.weight"].half())
        assert torch.equal(L["wgu"][1::2], merged[p + "mlp.gate_proj.weight"].half())
        assert torch.equal(L["wdown"], merged[p + "mlp.down_proj.weight"].half())
        assert torch.equal(L["ln1"], merged[p + "input_layernorm.weight"]) and not torch.equal(L["ln1"], base[p + "input_layernorm.weight"])
    assert torch.equal(m.norm, merged["model.norm.weight"])
    with pytest.raises(SeedxError):                                     # rank mismatch vs the configured r
        m.peft_config = lora.LoraConfig(r=8, lora_alpha=8)
        m.apply_peft_state_dict(ft)


def test_kv_page_allocator_and_page_table_rows():
    """host half of the paged KV cache: free-list accounting, growth of a slot's reservation, release on a fresh request, exhaustion"""
    import torch
    from seedx_b200 import synth
    from seedx_b200._lib import SeedxError
    from seedx_b200.llm import KVPageAllocator, LlamaForCausalLM
    a = KVPageAllocator(5)
    p = a.alloc(3)
    assert len(set(p)) == 3 and len(a.free) == 2
    with pytest.raises(SeedxError, match="KV cache exhausted"):
        a.alloc(3)
    a.release(p)
    assert sorted(a.free) == [0, 1, 2, 3, 4]
    cfg = dict(synth.TINY_LLAMA)
    m = LlamaForCausalLM(cfg, max_len=100, device="cpu", kv_page_size=16)
    m.load_state_dict(synth.llama_state_dict(cfg))
    m._alloc_state(2)
    assert m.pages_per_slot == 7 and m.kv_alloc.n_pages == 14 and tuple(m.kcache[0].shape) == (14, 16, cfg["hidden"])
    m.reserve_kv(0, 17, fresh=True)
    first = list(m.slot_pages[0])
    assert len(first) == 2 and m.page_table[0, :2].tolist() == first
    m.reserve_kv(1, 40, fresh=True)
    m.reserve_kv(0, 60)                                    # grows, keeps the pages (and cached rows) it already has
    assert m.slot_pages[0][:2] == first and len(m.slot_pages[0]) == 4 and m.page_table[0, :4].tolist() == m.slot_pages[0]
    assert not set(m.slot_pages[0]) & set(m.slot_pages[1])
    m.reserve_kv(0, 5, fresh=True)                         # new request in the slot: old pages returned first
    assert len(m.slot_pages[0]) == 1 and len(m.kv_alloc.free) + 1 + len(m.slot_pages[1]) == 14
    with pytest.raises(SeedxError, match="exceeds the KV cache"):
        m.reserve_kv(0, 101)
    with pytest.raises(SeedxError):
        LlamaForCausalLM(cfg, kv_page_size=48)
