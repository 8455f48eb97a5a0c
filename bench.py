#!/usr/bin/env python
"""bench.py — end-to-end images/sec of the SEED-X hot path on N B200s of one node (one process per GPU, replicas).

Workloads (BASELINE.json `configs`; `--workload`):
  i2i (default, the headline metric: 448x448 in -> 1024x1024 out; configs[2] = its de-tokenizer stage at batch 4)
      448^2 image (any-res '1x1' grid -> 2 ViT views) + 32-token prompt ending in <img>
      -> ViT-bigG -> LLaMA-13B prefill + 66 greedy tokens (65 of them forced by the image-token logits processor) -> output resampler
      -> ResamplerXLV2 -> 50 Euler steps x 2-way CFG SDXL UNet @128^2 latents -> VAE decode -> 1024^2 uint8 image; 4 requests per GPU.
  edit (configs[3]: SEED-X-Edit, 1024^2 source + edit prompt -> 1024^2 edited image, batch 8 over 8 GPUs = 1 request per GPU)
      as i2i up to the image features, then VAE encode of the 1024^2 source, 50 steps x 3-way CFG (150 UNet sample-forwards, 8-channel
      conv_in, sigma-space combine), VAE decode.
  anyres (configs[4]: dynamic-res multi-image, 2x2 grid of 448^2 tiles -> 5 ViT views, text + image, batch 32 over 8 GPUs = 4 per GPU)
      5 views -> prompt of ~370 tokens -> 128 free-running greedy text tokens -> the image span behind that answer -> 50 steps x 2-way CFG
      -> VAE decode.
  comprehension (configs[1]: 1 x 448^2 image + 32-token prompt -> 128 text tokens, batch 1; auxiliary tokens/s line, HBM-bound).
Weights: random-init at the full architecture sizes (no checkpoints offline).  Ranks are independent replicas (weak scaling), NCCL only
gathers the finished images.

Prints ONE JSON line (rank 0).  `value` = device-resident inputs; `e2e` = pinned-host inputs copied in and results copied out inside the
timed region.  `roofline` is for the dominant launch, the CUDA-graphed UNet sample-forward (6.75 TFLOP per sample, SURVEY.md A.4).
`cpu_baseline` / `--impl reference`: the CPU oracle (oracle/, the reference's PyTorch path restated) timed on the host cores, ONE UNIT PER
STAGE (a ViT view, LLaMA layers in prefill and in decode, a UNet sample-forward, a VAE decode / encode) and extrapolated to the workload by
the exact number of units the unmodified reference would execute (BASELINE.md §4); the per-stage CPU seconds are printed.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# analytic work per unit, TFLOP (SURVEY.md Appendix A.4 / BASELINE.md §3)
VIT_TFLOP_448, VIT_TFLOP_224 = 4.219, 1.011
VIT_POOL_TFLOP_448, VIT_POOL_TFLOP_224 = 0.118, 0.0476
UNET_TFLOP, VAE_DEC_TFLOP, VAE_ENC_TFLOP = 6.75, 10.47, 4.54
LLM_GFLOP_TOK = 25.7
LLM_GB_PER_TOKEN = 26.04
METRIC = "end-to-end images/sec (448x448 in -> 1024x1024 out)"

# what ONE request of a workload makes the UNMODIFIED reference execute (its own code path, /root/reference/src/inference/eval_*.py):
#   ViT views include the negative ViT(zeros) the reference recomputes on every adapter.generate call (adapter_modules.py:109-111),
#   every generated token is one decode step (the reference has no jump-forward), CFG branches are separate UNet samples.
WORKLOADS = {
    "i2i": dict(views=2, neg_views=1, text_tokens=0, branches=2, vae_enc=0, default_batch=4,
                name="seedx_i2i_448_to_1024", metric=METRIC),
    "edit": dict(views=2, neg_views=1, text_tokens=0, branches=3, vae_enc=1, default_batch=1,
                 name="seedx_edit_1024_to_1024 (BASELINE.json configs[3])",
                 metric="end-to-end images/sec (SEED-X-Edit: 1024x1024 source + edit prompt -> 1024x1024 edited image)"),
    "anyres": dict(views=5, neg_views=1, text_tokens=128, branches=2, vae_enc=0, default_batch=4,
                   name="seedx_anyres_2x2_text_and_image (BASELINE.json configs[4])",
                   metric="end-to-end images/sec (dynamic-res 2x2 grid = 5 x 448x448 views -> 128 text tokens + 1024x1024 image)"),
    "comprehension": dict(views=2, neg_views=0, text_tokens=128, branches=0, vae_enc=0, default_batch=1,
                          name="seedx_comprehension_448 (BASELINE.json configs[1])", metric="comprehension text tokens/sec"),
}
PROMPT_LEN = {2: 182, 5: 380}          # <s> [INST] + views x 66 span tokens + 32 text tokens + [/INST]\n + <img> (SeedXEngine.build_prompt, SynthTokenizer)
DUMP_BYTES = 64 * 10 ** 6               # --dump-outputs: bytes written in all, .npy headers included


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each array as out_dir/<name>.npy in float32 (uint8 pixels and token ids are exact in it).  When the arrays exceed
    DUMP_BYTES together, each is replaced by a sample of its flattened elements, in index order, drawn with a fixed seed and sized in
    proportion to the array: runs with the same arguments write the same elements, so two builds compare output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float32) for k, v in arrays.items()}
    budget = (DUMP_BYTES - 1024 * len(arrays)) // 4
    total = sum(a.size for a in arrays.values())
    for name, a in arrays.items():
        if total > budget:
            idx = np.random.default_rng(0).choice(a.size, a.size * budget // total, replace=False)
            a = a.reshape(-1)[np.sort(idx)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def unit_counts(workload, steps=50):
    """units per request the reference executes: (ViT views, prefill rows, decode steps, UNet sample-forwards, VAE decodes, VAE encodes)"""
    w = WORKLOADS[workload]
    P = PROMPT_LEN[w["views"]]
    if workload == "comprehension":
        return dict(vit_views=w["views"], prefill_rows=P, decode_steps=128, unet_forwards=0, vae_dec=0, vae_enc=0)
    dec = w["text_tokens"] + 66                              # free text, then <img_0..63> </img> and the step that ends the span
    return dict(vit_views=w["views"] + w["neg_views"], prefill_rows=P, decode_steps=dec, unet_forwards=w["branches"] * steps, vae_dec=1,
                vae_enc=w["vae_enc"])


def work_per_image_tflop(workload="i2i", steps=50):
    c = unit_counts(workload, steps)
    llm = (c["prefill_rows"] + c["decode_steps"]) * LLM_GFLOP_TOK / 1e3
    return c["vit_views"] * VIT_TFLOP_448 + llm + c["unet_forwards"] * UNET_TFLOP + c["vae_dec"] * VAE_DEC_TFLOP + c["vae_enc"] * VAE_ENC_TFLOP


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["bf16_tflops_sustained"], d["hbm_gbs"], "measured (MEASURED_PEAKS.json, sustained bf16 cuBLAS)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md: ~1.4 PFLOP/s sustained, 6.65 TB/s)"


def measured_traffic():
    """per-launch DRAM bytes from the committed ncu captures (profiles/r02_traffic.json, written by tools/summarize_traffic.py from the raw
    ncu CSVs next to it); None when no capture is committed for this batch size"""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    return json.load(open(p)) if os.path.exists(p) else {}


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx, self.rows, self.stop = gpu_index, [], threading.Event()
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(timeout=3)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(self.rows)}


def pick_threads():
    """Thread count for the CPU arm = the one that is actually fastest on this host: more threads than the container's real core budget
    (cgroup quota, SMT siblings) make torch's CPU GEMMs slower, not faster, so 'all the threads it can use' is calibrated on a 2048^3 fp32
    matmul over a ladder of candidates instead of taken from os.cpu_count()."""
    import torch
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cands = sorted({c for c in (4, 8, 16, 32, 64, 128, 256, avail) if 1 <= c <= avail}) or [1]
    a, b = torch.randn(2048, 2048), torch.randn(2048, 2048)
    best_c, best_rate = cands[0], 0.0
    for c in cands:
        torch.set_num_threads(c)
        a @ b
        t0 = time.time()
        for _ in range(2):
            a @ b
        rate = 2 * 2 * 2048 ** 3 / max(time.time() - t0, 1e-9)
        if rate > best_rate * 1.03:
            best_c, best_rate = c, rate
    torch.set_num_threads(best_c)
    return best_c, avail


# ------------------------------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle (reference restated, fp32 torch) timed one unit per stage on the host cores
# ------------------------------------------------------------------------------------------------------------------------------------------
class CpuUnits:
    """Builds the per-stage CPU problems lazily (random-init weights at the full widths, drawn on the host) and times ONE unit of each:
      vit       one 448^2 view through VIT_LAYERS of the 48 blocks + the attention pool  -> scaled to 48 blocks by FLOPs within the stage
      llm       LLM_LAYERS of the 40 LLaMA-13B layers + lm_head: prefill of P rows, then decode steps over the cache -> layers scaled x40/LLM_LAYERS
      unet      one SDXL UNet sample-forward at 128^2 latents, 64 x 2048 context, batch 1 (exactly the unit the reference runs 100-150x per image)
      vae_dec   one VAE decode 128^2 latent -> 1024^2;  vae_enc  one VAE encode of a 1024^2 image
    No stage's time is inferred from another stage's FLOP rate."""
    VIT_LAYERS, LLM_LAYERS = 12, 2

    def __init__(self, threads, log=None):
        import torch
        self.torch, self.threads, self.log = torch, threads, (log or (lambda *a: None))
        torch.set_num_threads(threads)
        self._cache = {}
        self.samples = {}            # stage -> list of seconds (first execution = warm-up when there are more)

    def _get(self, key, make):
        if key not in self._cache:
            t0 = time.time()
            self._cache[key] = make()
            self.log(f"cpu arm: built {key} in {time.time() - t0:.1f}s")
        return self._cache[key]

    def _time(self, stage, fn):
        t0 = time.time()
        with self.torch.no_grad():
            out = fn()
        self.samples.setdefault(stage, []).append(time.time() - t0)
        return out

    def seconds(self, stage):
        s = self.samples.get(stage, [])
        if not s:
            return None
        return statistics.mean(s[1:]) if len(s) > 1 else s[0]

    # ---- units
    def vit(self):
        from oracle import vit as ovit
        from seedx_b200 import synth
        L = self.VIT_LAYERS
        sd = self._get("vit", lambda: synth.vit_state_dict(width=1664, layers=L, heads=16, mlp_width=8192, output_dim=4096, n_queries=256, patch=14))
        x = self._get("vit_x", lambda: synth.image("bench_cpu_view", 1, 448))
        return self._time("vit", lambda: ovit.vit_forward(sd, x, 16))

    def llm(self, P):
        from oracle import llm as ollm
        from seedx_b200 import synth
        torch = self.torch
        cfg = dict(vocab=32330, hidden=5120, layers=self.LLM_LAYERS, heads=40, ffn=13824, eps=1e-5)
        sd = self._get("llm", lambda: synth.llama_state_dict(cfg))
        emb = self._get(f"llm_x{P}", lambda: synth.randn("bench_cpu_llm_x", (P, 5120)))
        _, _, cache = self._time("llm_prefill", lambda: ollm.llama_forward(sd, cfg, emb, 0, None))
        one = emb[:1]

        def dec():
            c = cache
            for i in range(2):
                _, _, c = ollm.llama_forward(sd, cfg, one, P + i, c)
        self._time("llm_decode2", dec)
        w, h = sd["lm_head.weight"], emb
        self._time("llm_head_prefill", lambda: h @ w.t())
        self._time("llm_head_decode", lambda: one @ w.t())
        self.P = P

    def unet(self, in_channels=4):
        from oracle import sdxl as osd
        from seedx_b200 import synth
        cfg = dict(synth.SDXL_UNET, in_channels=in_channels)
        sd = self._get(f"unet{in_channels}", lambda: synth.unet_state_dict(cfg))
        torch = self.torch
        x, ctx, te = synth.randn("bench_cpu_ux", (1, in_channels, 128, 128)), synth.randn("bench_cpu_uc", (1, 64, 2048)), synth.randn("bench_cpu_ut", (1, 1280))
        tid = torch.tensor([[1024.0, 1024.0, 0.0, 0.0, 1024.0, 1024.0]])
        return self._time("unet", lambda: osd.unet_forward(sd, cfg, x, 601.0, ctx, te, tid))

    def vae_dec(self):
        from oracle import sdxl as osd
        from seedx_b200 import synth
        sd = self._get("vae", lambda: synth.vae_state_dict(synth.SDXL_VAE))
        z = synth.randn("bench_cpu_z", (1, 4, 128, 128))
        return self._time("vae_dec", lambda: osd.vae_decode(sd, synth.SDXL_VAE, z / 0.13025))

    def vae_enc(self):
        from oracle import sdxl as osd
        from seedx_b200 import synth
        sd = self._get("vae", lambda: synth.vae_state_dict(synth.SDXL_VAE))
        x = synth.randn("bench_cpu_img", (1, 3, 1024, 1024), 0.5).clamp(-1, 1)
        return self._time("vae_enc", lambda: osd.vae_encode_mode(sd, synth.SDXL_VAE, x))

    # ---- extrapolation by exact unit counts
    def per_request_seconds(self, workload, steps=50):
        c = unit_counts(workload, steps)
        s = self.seconds
        out = {}
        if s("vit") is not None:
            flop_unit = (VIT_TFLOP_448 - VIT_POOL_TFLOP_448) * self.VIT_LAYERS / 48 + VIT_POOL_TFLOP_448
            out["vit"] = c["vit_views"] * s("vit") * VIT_TFLOP_448 / flop_unit
        if s("llm_prefill") is not None:
            k = 40 / self.LLM_LAYERS
            rows = c["prefill_rows"] / self.P
            out["llm_prefill"] = ((s("llm_prefill") - s("llm_head_prefill")) * k + s("llm_head_prefill")) * rows
            out["llm_decode"] = c["decode_steps"] * ((s("llm_decode2") / 2 - s("llm_head_decode")) * k + s("llm_head_decode"))
        if c["unet_forwards"] and s("unet") is not None:
            out["unet"] = c["unet_forwards"] * s("unet")
        if c["vae_dec"] and s("vae_dec") is not None:
            out["vae_dec"] = c["vae_dec"] * s("vae_dec")
        if c["vae_enc"] and s("vae_enc") is not None:
            out["vae_enc"] = c["vae_enc"] * s("vae_enc")
        return out, c

    def stages_for(self, workload):
        w = WORKLOADS[workload]
        st = ["unet", "vae_dec"] if w["branches"] else []
        if w["vae_enc"]:
            st.append("vae_enc")
        return st + ["vit", "llm"]

    def run_unit(self, stage, workload):
        w = WORKLOADS[workload]
        if stage == "llm":
            self.llm(PROMPT_LEN[w["views"]])
        elif stage == "unet":
            self.unet(8 if workload == "edit" else 4)
        else:
            getattr(self, stage)()

    def report(self, workload, steps=50):
        per, counts = self.per_request_seconds(workload, steps)
        total = sum(per.values())
        unit_s = {k: self.seconds(k) for k in self.samples}
        sample = ("oracle (reference PyTorch path restated, fp32 torch CPU) on %d threads, one timed unit per stage: " % self.threads +
                  "; ".join(f"{k} {v:.2f}s" for k, v in unit_s.items()) +
                  f" [vit = one 448^2 view, {self.VIT_LAYERS}/48 blocks + pool; llm = {self.LLM_LAYERS}/40 layers + lm_head, prefill of {getattr(self, 'P', 0)} rows and "
                  "2 decode steps; unet = one full sample-forward; vae = one full 1024^2 decode/encode]; extrapolated by the unit counts the unmodified "
                  "reference executes per request " + json.dumps(counts) + " -> per-request CPU seconds " + json.dumps({k: round(v, 1) for k, v in per.items()}))
        return total, per, counts, unit_s, sample


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (oracle port of its PyTorch modules) on the host cores.  Each step
    times ONE stage unit, rotating over the stages of the workload (a full UNet sample-forward alone is ~15 s of CPU, so a step cannot hold
    one unit of every stage and still leave K + W steps within minutes); the line's value extrapolates by exact unit counts."""
    cores, avail = pick_threads()
    log = lambda *a: print("[bench ref]", *a, file=sys.stderr, flush=True)  # noqa: E731
    cu = CpuUnits(cores, log)
    wl = args.workload
    stages = cu.stages_for(wl)
    step_s = []
    for i in range(args.warmup + args.steps):
        t0 = time.time()
        cu.run_unit(stages[i % len(stages)], wl)
        if i >= args.warmup:
            step_s.append(time.time() - t0)
    for st in stages:                       # K + W smaller than the number of stages: every stage still gets its one unit
        key = "llm_prefill" if st == "llm" else st
        if not cu.samples.get(key):
            cu.run_unit(st, wl)
    total, per, counts, unit_s, sample = cu.report(wl, args.denoise_steps)
    if wl == "comprehension":
        value, unit = 128 / total, "tokens/s"
    else:
        value, unit = 1.0 / total, "images/s"
    line = {"impl": "reference", "metric": WORKLOADS[wl]["metric"], "value": value, "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": statistics.mean(step_s) * 1e3 if step_s else None, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOADS[wl]["name"] + " — CPU arm: each step = one stage unit (rotation " + "/".join(stages) + "), see cpu_baseline.sample",
                       "denoise_steps": args.denoise_steps},
            "cpu_stage_seconds_per_request": per, "cpu_unit_seconds": unit_s, "unit_counts_per_request": counts,
            "cpu_baseline": {"value": value, "unit": unit, "cores": cores, "kind": "port", "sample": sample, "schedulable_cpus": avail},
            "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------------------------------
# comprehension workload (auxiliary line)
# ------------------------------------------------------------------------------------------------------------------------------------------
def run_comprehension(args, eng, rank, world, peaks_, cpu_base):
    """--workload comprehension = BASELINE.json configs[1]: 1 x 448^2 image (any-res 1x1 -> 2 ViT views) + 32-token prompt -> 128 greedy text tokens,
    batch 1 per GPU (EOS suppressed so every step decodes exactly 128 tokens).  Auxiliary line: tokens/s, ms per token, decode HBM roofline."""
    import torch
    from seedx_b200 import _lib, synth, trace
    from seedx_b200 import dist as sdist
    tensor_peak, hbm_peak, peak_src = peaks_
    new_tok = 128
    views_host = synth.image(f"bench_cmp_views_rank{rank}", 2, 448).pin_memory()
    views_dev = views_host.cuda()
    patch_pos = torch.tensor([[0.5, 0.5], [0.5, 0.5]])
    text_ids = torch.randint(3, eng.tok.base, (32,), generator=torch.Generator().manual_seed(4321 + rank)).tolist()
    ids, mask = eng.build_prompt(2, text_ids, force_image=False)
    P = int(ids.numel())

    def step(e2e):
        v = views_host.cuda(non_blocking=True) if e2e else views_dev
        feats = eng.vit(v)
        trace.mark("vit")
        req = dict(input_ids=ids.unsqueeze(0), image_embeds=feats, embeds_cmp_mask=torch.ones((2, 64), dtype=torch.bool), ids_cmp_mask=mask.unsqueeze(0),
                   patch_positions=patch_pos)
        out = eng.agent.generate_batch(eng.tok, [req], max_new_tokens=new_tok, suppress_eos=True)[0]   # reads the ids back to the host (d2h)
        return out

    def timed(e2e):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = _lib.launch_count()
        e0.record()
        for _ in range(args.steps):
            out = step(e2e)
        e1.record()
        torch.cuda.synchronize()
        assert len(out["ids"]) == new_tok
        return sdist.max_over_ranks(e0.elapsed_time(e1), "cuda"), _lib.launch_count() - n0, out

    for _ in range(args.warmup):
        step(False)
    with ClockSampler(int(os.environ.get("LOCAL_RANK", "0"))) as cs:
        ms_dev, launches, last = timed(False)
        ms_e2e, _, _ = timed(True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"text_ids": last["ids"]})
    trace.enable(True)
    trace.mark("start")
    step(False)
    detail = trace.summary()
    trace.enable(False)
    if rank == 0:
        toks = world * new_tok * args.steps
        dec_ms = detail.get("llm.decode", 0.0)
        gb = LLM_GB_PER_TOKEN * (new_tok - 1)
        print(json.dumps({
            "metric": "comprehension text tokens/sec (1x448^2 image + 32-token prompt -> 128 greedy tokens, batch 1 per GPU)", "value": toks / (ms_dev / 1e3),
            "unit": "tokens/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": "seedx_comprehension_448 (BASELINE.json configs[1]): prompt %d tokens incl. 2 x 64 image rows, 128 new tokens, EOS suppressed" % P,
                       "weights": "random-init, full sizes", "l2": "26 GB of weights per token step exceed the 126 MB L2"},
            "stage_detail_ms": detail,
            "e2e": {"value": toks / (ms_e2e / 1e3), "unit": "tokens/s", "h2d_bytes_per_step": views_host.numel() * 4 + P * 8,
                    "d2h_bytes_per_step": (P + new_tok) * 4, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches, "clocks": cs.summary(),
            "roofline": {"bound": "hbm", "kernel": "CUDA-graph replay of one decode step (gemv_mma_kernel = 84 % of it)", "achieved": gb / (dec_ms / 1e3) if dec_ms else None,
                         "peak": hbm_peak, "unit": "GB/s", "frac": gb / (dec_ms / 1e3) / hbm_peak if dec_ms else None,
                         "traffic": measured_traffic().get("decode_step_bytes"),
                         "ms_per_token": dec_ms / (new_tok - 1), "bytes_per_token_gb": LLM_GB_PER_TOKEN, "peak_source": peak_src},
            "cpu_baseline": cpu_base}))


# ------------------------------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=int(os.environ.get("SEEDX_BENCH_BATCH", "0")), help="requests per GPU per step (0 = the workload's default)")
    ap.add_argument("--denoise-steps", type=int, default=50)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--small", action="store_true", help="debug: tiny models (NOT a valid benchmark)")
    ap.add_argument("--workload", default="i2i", choices=sorted(WORKLOADS),
                    help="i2i (default, the headline metric) | edit (configs[3]) | anyres (configs[4]) | comprehension (configs[1], tokens/s)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step of the headline window returned (rank 0: images, text token ids) "
                         "as DIR/<name>.npy, float32, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours; the reference arm times single stage units")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if rank == 0:
            run_reference(args)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    torch.cuda.set_device(local)
    torch.manual_seed(0)            # the denoise loop draws its latent noise from the default generators: same arguments, same inputs
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from seedx_b200 import _lib, synth
    from seedx_b200 import dist as sdist
    from seedx_b200.engine import SeedXEngine
    log = (lambda *a: print("[bench]", *a, file=sys.stderr, flush=True)) if rank == 0 else None
    tensor_peak, hbm_peak, peak_src = peaks()
    wl = args.workload
    W = WORKLOADS[wl]
    B = args.batch or W["default_batch"]

    # ---- CPU baseline first (rank 0, N=1): one oracle unit per stage on the host cores (bounded: ~40 s of CPU work + weight draws) ------------
    cpu_base = None
    do_cpu = (world == 1 and rank == 0 and not args.no_cpu_baseline and not args.small)
    if do_cpu:
        cores, avail = pick_threads()
        cu = CpuUnits(cores, log)
        for st in cu.stages_for(wl):
            cu.run_unit(st, wl)
        total, per, counts, unit_s, sample = cu.report(wl, args.denoise_steps)
        v = (128 / total) if wl == "comprehension" else (1.0 / total)
        cpu_base = {"value": v, "unit": "tokens/s" if wl == "comprehension" else "images/s", "cores": cores, "kind": "port", "sample": sample,
                    "cpu_stage_seconds_per_request": per, "cpu_unit_seconds": unit_s, "unit_counts_per_request": counts, "schedulable_cpus": avail}
        log(f"cpu baseline: {json.dumps({k: round(x, 2) for k, x in unit_s.items()})} -> {total:.0f} CPU-seconds per request on {cores} threads")
        del cu

    if args.small:
        eng = SeedXEngine(vit_cfg=dict(width=208, layers=2, heads=2, mlp_width=520, output_dim=256, n_queries=256, patch=14),
                          llm_cfg=synth.TINY_LLAMA, unet_cfg=dict(synth.TINY_UNET, cross_attention_dim=256, text_embed_dim=160),
                          vae_cfg=synth.TINY_VAE, rxl_cfg=dict(synth.TINY_RESAMPLER_XL, embedding_dim=256, output1_dim=96, output2_dim=160),
                          log=log, edit=(wl == "edit"))
    else:
        eng = SeedXEngine(log=log, edit=(wl == "edit"))

    if wl == "comprehension":
        run_comprehension(args, eng, rank, world, (tensor_peak, hbm_peak, peak_src), cpu_base)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    n_views = W["views"]
    branches = W["branches"]
    # ---- synthetic inputs: post-transform views in pinned host memory + device-resident copies ------------------------------
    views_host = synth.image(f"bench_views_rank{rank}", B * n_views, 448).pin_memory()
    views_dev = views_host.cuda()
    if n_views == 5:     # any-res 2x2 grid (any_res.py:193-199): the 4 tiles at ((i + .5) / 2, (j + .5) / 2), then the resized whole image at (.5, .5)
        pp1 = [[0.25, 0.25], [0.75, 0.25], [0.25, 0.75], [0.75, 0.75], [0.5, 0.5]]
    else:
        pp1 = [[0.5, 0.5], [0.5, 0.5]]
    patch_pos = torch.tensor(pp1 * B)
    g = torch.Generator().manual_seed(1234 + rank)
    text_ids = [torch.randint(3, eng.tok.base, (32,), generator=g).tolist() for _ in range(B)]
    out_host = torch.empty((B, 1024, 1024, 3), dtype=torch.uint8).pin_memory() if not args.small else None
    h2d_bytes = views_host.numel() * 4 + B * 32 * 8
    d2h_bytes = B * 1024 * 1024 * 3
    src_host = src_dev = None
    if wl == "edit":
        src_host = synth.randn(f"bench_src_rank{rank}", (B, 3, 1024, 1024) if not args.small else (B, 3, 256, 256), 0.5).clamp_(-1, 1).pin_memory()
        src_dev = src_host.cuda()
        h2d_bytes += src_host.numel() * 4
    if W["text_tokens"]:
        d2h_bytes += B * W["text_tokens"] * 4
    gather_buf = None

    def step(e2e):
        v = views_host.cuda(non_blocking=True) if e2e else views_dev
        src = None
        if wl == "edit":
            src = src_host.cuda(non_blocking=True) if e2e else src_dev
        u8 = eng.generate(v, patch_pos, text_ids, steps=args.denoise_steps, n_views=n_views, source_images=src, text_tokens=W["text_tokens"])
        nonlocal gather_buf
        if world > 1:                                  # the only collective: gather finished images on every rank (NCCL / NVLink)
            gather_buf = sdist.gather_images(u8, gather_buf)
        if e2e:
            if out_host is not None:
                out_host.copy_(u8, non_blocking=True)
            else:
                u8.cpu()
        return u8

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(e2e=(i % 2 == 1))
        if log:
            log(f"warmup {i}: {eng.stage_ms()}")
    sync()

    def timed(e2e, keep=False):
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = _lib.launch_count()
        stages = []
        e0.record()
        for _ in range(args.steps):
            u8 = step(e2e)
            stages.append(eng._events)
        e1.record()
        sync()
        if keep:                                       # outside the timed window, before the next step can reuse the buffers
            kept["images"] = u8.cpu().numpy()
            if W["text_tokens"]:
                kept["text_ids"] = eng.last_text_ids
        ms = sdist.max_over_ranks(e0.elapsed_time(e1), "cuda")
        st = {k: statistics.mean(a.elapsed_time(b) for (a, b) in [(ev[i], ev[i + 1]) for ev in stages])
              for i, k in enumerate(("vit_ms", "llm_ms", "detok_ms"))}
        return ms, _lib.launch_count() - n0, st

    kept = {}
    if rank == 0:       # one nvidia-smi poller per job (8 of them would only add host noise); rank 0's GPU stands for the box
        with ClockSampler(local) as cs:
            ms_dev, launches, stages = timed(e2e=False, keep=bool(args.dump_outputs))
            ms_e2e, _, _ = timed(e2e=True)
        clocks = cs.summary()
        if kept:
            dump_outputs(args.dump_outputs, kept)
    else:
        ms_dev, launches, stages = timed(e2e=False)
        ms_e2e, _, _ = timed(e2e=True)
        clocks = None
    # one extra untimed step with section marks on (seedx_b200.trace): where the step goes, stage by stage
    from seedx_b200 import trace
    trace.enable(True)
    step(e2e=False)
    detail = trace.summary()
    # decode probe (i2i / edit): the bench prompt ends in <img>, so its 65 forced image tokens ride through the prefill pass (jump-forward) and the
    # step has almost no token loop left; the HBM-bound decode path is therefore timed separately on 64 free-running token steps of B lock-step
    # sequences (64-token random prompts, EOS suppressed) — untimed for the headline, reported in stage_roofline.llm_decode.  The anyres workload
    # has 128 free-running tokens inside its timed step: its llm_decode figure comes from the step itself.
    decode_step_ms = None
    if not args.small and not W["text_tokens"]:
        trace.enable(True)
        pg = torch.Generator().manual_seed(99 + rank)
        p_ids = [torch.randint(3, eng.tok.base, (64,), generator=pg) for _ in range(B)]
        p_emb = [eng.llm.get_input_embeddings()(i)[0] for i in p_ids]
        eng.llm.generate_greedy_batch(p_ids, p_emb, img_ids=None, max_new_tokens=3, eos_id=None, suppress_eos=True)   # captures this rule's decode graph
        trace.enable(True)
        eng.llm.generate_greedy_batch(p_ids, p_emb, img_ids=None, max_new_tokens=65, eos_id=None, suppress_eos=True)
        decode_step_ms = trace.summary().get("llm.decode", 0.0) / 64
    trace.enable(False)
    # transparency: the same timed loop with jump-forward off (every forced image token takes its own decode step, as in the reference)
    token_loop = None
    if world == 1 and not args.small and eng.llm.jump_forward and wl == "i2i":
        try:
            eng.llm.jump_forward = False
            step(e2e=False)
            ms_tl, _, st_tl = timed(e2e=False)
            token_loop = {"value": B * args.steps / (ms_tl / 1e3), "unit": "images/s", "ms_per_step": ms_tl / args.steps, "stage_ms_per_step": st_tl,
                          "note": "SEEDX_JUMP_FORWARD=0 behaviour: the 65 forced image tokens decoded one step at a time"}
        except Exception as exc:                          # never let the extra measurement take the headline down
            token_loop = {"error": repr(exc)}
        finally:
            eng.llm.jump_forward = True

    if rank == 0:
        imgs = world * B * args.steps
        value = imgs / (ms_dev / 1e3)
        e2e_v = imgs / (ms_e2e / 1e3)
        traffic = measured_traffic()
        # dominant launch: the CUDA-graphed UNet sample-forward (branches x B samples per launch, 50 launches per step), timed live here with
        # CUDA events on the launching stream
        loop = next(iter(eng.adapter._loops.values()))
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10
        e0.record()
        for _ in range(reps):
            loop.graph.replay()
        e1.record()
        torch.cuda.synchronize()
        unet_ms = e0.elapsed_time(e1) / reps
        n_samples = branches * B
        achieved = UNET_TFLOP * n_samples / (unet_ms / 1e3) if not args.small else None
        # the dominant kernel's dominant shape, timed alone with CUDA events on the launching stream: gemm_tc_kernel<256,2> on the GEGLU
        # projection of the UNet feed-forward (60 launches per forward = 16 % of it, the largest single line of the launch list); three
        # operand sets (393 MB) rotate so that no launch finds its inputs in the 126 MB L2
        dom = None
        if not args.small:
            from seedx_b200 import ops
            Mg, Ng, Kg = n_samples * 1024, 10240, 1280
            As = [torch.randn(Mg, Kg, device="cuda").half() for _ in range(3)]
            Ws = [(torch.randn(Ng, Kg, device="cuda") * 0.03).half() for _ in range(3)]
            Os = [torch.empty(Mg, Ng // 2, device="cuda", dtype=torch.float16) for _ in range(3)]
            gb = torch.randn(Ng, device="cuda")
            for j in range(3):
                ops.gemm(As[j], Ws[j], out=Os[j], bias=gb, act=ops.ACT_GELU, gated=True)
            torch.cuda.synchronize()
            n_l = 30
            e0.record()
            for j in range(n_l):
                ops.gemm(As[j % 3], Ws[j % 3], out=Os[j % 3], bias=gb, act=ops.ACT_GELU, gated=True)
            e1.record()
            torch.cuda.synchronize()
            us = e0.elapsed_time(e1) * 1e3 / n_l
            fl = 2.0 * Mg * Ng * Kg
            tkey = f"geglu_gemm_M{Mg}_bytes"
            dom = {"kernel": "gemm_tc_kernel<256,2> (tcgen05 cta_group::2), GEGLU projection M=%d N=%d K=%d, bias + GELU gating fused" % (Mg, Ng, Kg),
                   "launch_us": us, "achieved": fl / us / 1e6, "unit": "TFLOP/s", "peak": tensor_peak, "frac": fl / us / 1e6 / tensor_peak,
                   "algorithmic_bytes": 2 * (Mg * Kg + Ng * Kg + Mg * Ng // 2), "traffic": traffic.get(tkey),
                   "traffic_source": traffic.get("source") if traffic.get(tkey) is not None else None}
            del As, Ws, Os
        # per-stage achieved rate against the roofline that bounds the stage (SURVEY.md §8d), from the marked extra step
        P = int(eng.build_prompt(n_views, text_ids[0])[0].numel())
        new_tok = 66

        def tens(tflop, ms):
            return {"bound": "tensor", "achieved": tflop / (ms / 1e3), "unit": "TFLOP/s", "peak": tensor_peak, "frac": tflop / (ms / 1e3) / tensor_peak,
                    "ms": ms}
        stage_roof = None
        if not args.small and detail:
            tt = W["text_tokens"]
            if tt:       # two prefill passes: the prompt, then prompt + answer + the forced image span
                rows = B * (P - 1) + B * (P + tt + new_tok - 1)
                dec_ms, n_dec = detail.get("llm.decode", 0.0), tt - 1
                decode_step_ms = dec_ms / max(n_dec, 1)
            else:
                rows = B * (P + new_tok - 1)
                dec_ms, n_dec = decode_step_ms * 64, 64
            gbs = LLM_GB_PER_TOKEN * n_dec
            stage_roof = {
                "vit": tens(B * n_views * VIT_TFLOP_448, detail["vit"]),
                "llm_prefill": dict(tens(rows * LLM_GFLOP_TOK / 1e3, detail["llm.prefill"]), prompt_len=P, rows=rows,
                                    note="rows per request = prompt + the 65 forced image tokens (jump-forward); all requests of a step share one "
                                         "pass over the weights" + ("; anyres: a second pass re-reads prompt + the 128-token answer" if tt else "")),
                "llm_decode": {"bound": "hbm", "achieved": gbs / (dec_ms / 1e3), "unit": "GB/s", "peak": hbm_peak, "frac": gbs / (dec_ms / 1e3) / hbm_peak,
                               "ms": dec_ms, "ms_per_token_step": decode_step_ms, "sequences_in_lock_step": B, "bytes_per_step_gb": LLM_GB_PER_TOKEN,
                               "note": ("the %d free-running token steps inside the timed step" % n_dec) if tt else
                                       ("probe outside the timed step: 64 free-running token steps (the step's own forced image tokens are "
                                        "teacher-forced rows of the prefill pass); token loop left inside the step: %.1f ms" % detail.get("llm.decode", 0.0))},
                "unet_denoise_loop": tens(n_samples * args.denoise_steps * UNET_TFLOP, detail["detok.denoise_loop"]),
                "vae_decode": tens(B * VAE_DEC_TFLOP, detail["detok.vae_decode"]),
            }
            if wl == "edit":
                stage_roof["vae_encode"] = tens(B * VAE_ENC_TFLOP, detail["detok.vae_encode"])
        # work per image as THIS engine executes it (negative ViT(zeros) cached, forced tokens as prefill rows) for the pipeline fraction
        own_tflop = (n_views * VIT_TFLOP_448 + (P + new_tok + (W["text_tokens"] * 2 + P if W["text_tokens"] else 0)) * LLM_GFLOP_TOK / 1e3 +
                     branches * args.denoise_steps * UNET_TFLOP + VAE_DEC_TFLOP + W["vae_enc"] * VAE_ENC_TFLOP)
        desc = {"i2i": "per GPU %d requests/step, each 1x448^2 image (any-res 1x1 -> 2 ViT views) + 32-token prompt -> ViT-bigG -> LLaMA-13B prefill + 66 greedy "
                       "tokens (65 forced by the image-token logits processor: teacher-forced rows of the prefill pass, results identical to token-by-token "
                       "decoding; SEEDX_JUMP_FORWARD=0 restores the loop) -> ResamplerXLV2 -> %d Euler steps x 2-way CFG SDXL UNet -> VAE decode -> 1024^2 uint8",
                "edit": "per GPU %d request(s)/step, each 1024^2 source image (448^2 any-res 1x1 -> 2 ViT views for the agent) + 32-token edit prompt -> ViT-bigG -> "
                        "LLaMA-13B (image span as in i2i) -> ResamplerXLV2 -> VAE encode of the source -> %d Euler steps x 3-way CFG (text/image/uncond, sigma space) "
                        "SDXL UNet with 8-channel conv_in -> VAE decode -> 1024^2 uint8",
                "anyres": "per GPU %d requests/step, each a 2x2 any-res grid (5 x 448^2 ViT views, patch positions) + 32-token prompt (P = 373) -> 128 free-running greedy "
                          "text tokens -> <img> span behind the answer (second prefill pass, 65 forced rows) -> ResamplerXLV2 -> %d Euler steps x 2-way CFG -> VAE "
                          "decode -> 1024^2 uint8"}[wl] % (B, args.denoise_steps)
        line = {
            "metric": W["metric"], "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16",
            "data": "synthetic",
            "config": {"workload": W["name"] + ": " + desc,
                       "requests_per_gpu": B, "denoise_steps": args.denoise_steps, "parallelism": f"replicas x{world} (one request set per rank)",
                       "l2": "working set (35 GB fp16 weights/GPU) exceeds the 126 MB L2; no explicit flush", "weights": "random-init, full sizes",
                       "small_debug_models": bool(args.small)},
            "stage_ms_per_step": stages,
            "stage_detail_ms": detail,
            "stage_roofline": stage_roof,
            "without_jump_forward": token_loop,
            "e2e": {"value": e2e_v, "unit": "images/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": {"bound": "tensor",
                         "kernel": "CUDA-graph launch of one UNet sample-forward (%d samples): gemm_tc_kernel (GEMM + implicit-GEMM conv) and tcgen05 attention, "
                                   "per-kernel shares and DRAM bytes in profiles/r02_unet_forward_launches_*.csv / .md" % n_samples,
                         "achieved": achieved, "peak": tensor_peak, "unit": "TFLOP/s", "frac": (achieved / tensor_peak) if achieved else None,
                         "dominant_kernel": dom, "traffic": traffic.get(f"unet_forward_{n_samples}samples_bytes"),
                         "traffic_source": traffic.get("source") if traffic.get(f"unet_forward_{n_samples}samples_bytes") is not None else None,
                         "peak_source": peak_src, "flop_per_launch": UNET_TFLOP * n_samples * 1e12,
                         "launch_ms": unet_ms, "graph_kernels": getattr(loop, "graph_kernels", None),
                         "work_per_image_tflop": own_tflop, "reference_work_per_image_tflop": work_per_image_tflop(wl, args.denoise_steps),
                         "pipeline_frac": (value / world) * own_tflop / tensor_peak},
            "cpu_baseline": cpu_base,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()          # rank 0 is still measuring the roofline launches: nobody tears the communicator down before it is done
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
