#!/usr/bin/env python
"""Benchmark of the parallel-denoising hot path (BASELINE.json metric):
denoised tokens/sec (text+image) per 512x512 @ 64-step sample, variant A 8B, cfg_img=4 (BASELINE configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference ...                            # the reference algorithm on the host CPU (oracle port)
    python bench.py --dump-outputs DIR ...                          # also writes what the last timed sample computed (.npy)

One "step" = one full sample = one generate_ti2ti call: 128 denoising iterations, 192 transformer forwards
(128 conditional + 64 unconditional-image), 128 text steps, 64 image steps -> 1280 denoised tokens.
Under torchrun (N > 1) every rank denoises its own independent prompt (replicas, no data-path collective): weak scaling.
Prints ONE JSON line on rank 0. Timing: CUDA events on the launching stream, barrier + synchronize on both sides,
max over ranks. Weights (16.2 GB) are re-read from HBM every forward, far beyond the 126 MB L2, so no L2 flush is needed.
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

TOKENS_PER_SAMPLE = 1024 + 256
MASK, NL, BOA, BOI, EOI, EOA = 126336, 126084, 126354, 126349, 126350, 126355
TEXT_VOCAB, CODEBOOK = 126356, 8192

MODEL_8B = dict(d_model=4096, n_heads=32, n_layers=32, mlp_hidden_size=12288, vocab_size=134656, max_sequence_length=2432)
MODEL_TINY = dict(d_model=256, n_heads=2, n_layers=2, mlp_hidden_size=512, vocab_size=134656, max_sequence_length=2432)
GEN = dict(text_steps=128, timesteps=64, text_gen_length=256, text_block_length=32, temperature=1.0, text_temperature=0.0,
           cfg_scale=0.0, cfg_img=4.0)  # README.md:101-117 of the reference


def synthetic_layout(seed: int, prompt_len: int = 40, grid: int = 32, text_len: int = 256):
    """SURVEY.md 8d synthetic input A: L = P + 2374 = 2414 at P = 40 (structure of A/inference.py:129-156)."""
    g = torch.Generator().manual_seed(seed)
    prompt = torch.randint(0, 126000, (prompt_len,), generator=g).tolist()
    img_in = torch.randint(TEXT_VOCAB, TEXT_VOCAB + CODEBOOK, (grid * grid,), generator=g).tolist()
    img = [BOI]
    for r in range(grid):
        img += img_in[r * grid:(r + 1) * grid] + [NL]
    img += [EOI]
    con = prompt[:-1] + img + prompt[-1:]
    pred = [BOA, BOI]
    for _ in range(grid):
        pred += [MASK] * grid + [NL]
    pred += [EOI] + [MASK] * text_len + [EOA]
    ids = con + pred
    image_start = len(con) + 2
    text_start = image_start + grid * (grid + 1) + 1
    unc_prompt = torch.randint(0, 126000, (3,), generator=g).tolist()
    return dict(input_ids=torch.tensor([ids]), text_start=text_start, text_end=text_start + text_len,
                image_start=image_start, seq_len=grid * grid, newline_every=grid,
                uncon_text=torch.tensor([unc_prompt[:-1] + img + unc_prompt[-1:]]), uncon_image=torch.tensor([prompt]))


def quiet():
    return contextlib.redirect_stdout(io.StringIO())


# ------------------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.p = gpu_index, None

    def start(self):
        try:
            self.f = tempfile.NamedTemporaryFile("w+", prefix="mmdp_clocks_", suffix=".csv")
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                       "-i", str(self.idx)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.seek(0)
        lines = self.f.readlines()
        self.f.close()  # removes the file
        sm, mx, reasons, power = [], [], set(), []
        for line in lines:
            c = [x.strip() for x in line.split(",")]
            if len(c) < 8:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2])); power.append(float(c[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        loaded = [s for s, p in zip(sm, power) if p > 0.5 * max(power)] or sm
        return {"sm_mhz": statistics.median(loaded), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "power_w_max": max(power), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference algorithm (oracle port) on the host cores, bounded sample, extrapolated by exact counts
# ------------------------------------------------------------------------------------------------------------------
def host_cpu_info():
    """CPU model string, physical cores, logical CPUs of the box this runs on."""
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    logical = os.cpu_count() or 1
    try:
        import psutil
        physical = psutil.cpu_count(logical=False) or logical
    except Exception:
        physical = logical
    try:
        usable = len(os.sched_getaffinity(0))
    except Exception:
        usable = logical
    return {"model": model, "physical_cores": int(min(physical, usable)), "logical_cpus": int(logical), "usable_cpus": int(usable)}


def cpu_reference_sample(model_cfg: dict, reps: int = 3):
    """Times the path's CPU restatement (oracle/, the port of the reference; /root/reference is not on the GPU box) at
    the full BASELINE shapes on a bounded sample and extrapolates to one full sample with the exact operation counts:
      192 forwards x n_layers block-forwards  +  128 text-row heads  +  128 image-col heads (64 cond + 64 uncond)
      + 128 text steps + 64 image steps.
    Protocol (round-1 numbers swung 5x between boxes with one cold repetition on all logical CPUs): threads are swept over
    {physical cores, half, quarter} (never more than the physical cores), every setting gets one warm-up and `reps` timed
    block forwards, the MEDIAN of the best setting is used, and the CPU model / core counts are reported."""
    from oracle import llada, sampling as S
    info = host_cpu_info()
    phys = max(1, info["physical_cores"])
    cfg = llada.make_config(**model_cfg)
    d, ff, V, L = cfg.d_model, cfg.mlp_hidden_size, cfg.vocab_size, 2414
    g = torch.Generator().manual_seed(0)
    rnd = lambda *s, std=0.02: (torch.randn(*s, generator=g) * std).to(torch.bfloat16)
    p = "b."
    w = {p + "q_proj.weight": rnd(d, d), p + "k_proj.weight": rnd(d, d), p + "v_proj.weight": rnd(d, d),
         p + "attn_out.weight": rnd(d, d), p + "ff_proj.weight": rnd(ff, d), p + "up_proj.weight": rnd(ff, d),
         p + "ff_out.weight": rnd(d, ff), p + "attn_norm.weight": torch.ones(d, dtype=torch.bfloat16),
         p + "ff_norm.weight": torch.ones(d, dtype=torch.bfloat16)}
    head = rnd(V, d)
    x = rnd(1, L, d, std=1.0)
    pos_sin, pos_cos = llada.rotary_tables(d // cfg.n_heads, cfg.rope_theta, L)

    def med(fn, n):
        ts = []
        for _ in range(n):
            t0 = time.perf_counter()
            r = fn()
            ts.append(time.perf_counter() - t0)
        return statistics.median(ts), r

    sweep = {}
    with torch.no_grad():
        for threads in sorted({phys, max(1, phys // 2), max(1, phys // 4)}, reverse=True):
            torch.set_num_threads(threads)
            llada.block_forward(x, w, p, cfg, pos_sin, pos_cos)  # warm-up (thread pool, oneDNN primitives)
            t, _ = med(lambda: llada.block_forward(x, w, p, cfg, pos_sin, pos_cos), reps)
            sweep[threads] = t
            if t > 20.0:  # a box this slow gets one thread setting only (keeps the arm bounded)
                break
        threads = min(sweep, key=sweep.get)
        t_block = sweep[threads]
        torch.set_num_threads(threads)
        y = llada.block_forward(x, w, p, cfg, pos_sin, pos_cos)
        xt = y[0, 2157:2413]
        torch.nn.functional.linear(xt, head)
        t_head_text, tl = med(lambda: torch.nn.functional.linear(xt, head), reps)
        xi = y[0, 1100:1100 + 1024]
        torch.nn.functional.linear(xi, head[TEXT_VOCAB:TEXT_VOCAB + CODEBOOK])
        t_head_img, il = med(lambda: torch.nn.functional.linear(xi, head[TEXT_VOCAB:TEXT_VOCAB + CODEBOOK]), reps)
        ids = torch.full((256,), MASK)
        S.text_step(tl, ids, MASK, 2)
        t_text, _ = med(lambda: S.text_step(tl, ids, MASK, 2), reps)
        vq = torch.full((1024,), -1)
        q = torch.empty(1024, CODEBOOK, dtype=torch.bfloat16).exponential_(1, generator=g)
        rn = torch.randn(1024, generator=g).to(torch.bfloat16)
        img = lambda: S.image_step("A", il, None, il.flip(0), 0.0, 4.0, vq, MASK, 600, 0.5, q, rn, CODEBOOK)
        img()
        t_img, _ = med(img, reps)
    n_layers = cfg.n_layers
    per_sample = 192 * n_layers * t_block + 128 * t_head_text + 128 * t_head_img + 128 * t_text + 64 * t_img
    return dict(tokens_per_s=TOKENS_PER_SAMPLE / per_sample, sec_per_sample=per_sample, cores=threads, cpu=info,
                thread_sweep_sec_per_block={str(k): round(v, 4) for k, v in sweep.items()},
                t_block=t_block, t_head_text=t_head_text, t_head_img=t_head_img, t_text_step=t_text, t_image_step=t_img,
                sample=f"median of {reps} block forwards (after 1 warm-up) of {192 * n_layers} per sample (d={d}, ff={ff}, L={L}) on {threads} threads "
                       f"(best of the sweep {sorted(sweep)}; {info['model']}, {info['physical_cores']} physical cores) + text/image heads + 1 text step "
                       f"+ 1 image step, extrapolated with the exact per-sample counts")


def gpu_eager_baseline(model_cfg: dict, device: str, lay: dict, seed: int = 1000):
    """The reference ALGORITHM in PyTorch eager on this GPU (BASELINE.md 4(iii), SURVEY 8d "the practical bar to beat"):
    the oracle port of LLaDAModel.forward + the generate_ti2ti step run with device='cuda' tensors - cuBLAS GEMMs, torch SDPA,
    ATen elementwise kernels, FULL LM head [L, V] like the reference. /root/reference itself is not on the GPU box, so the
    port stands in for it, which FAVOURS the baseline: its step has none of the reference's ~3 300 .item() syncs per image
    step and it skips the unused uncond_text forward. Timed: 4 text-only steps and 2 image steps (cond + uncond_image
    forwards) after one warm-up of each, extrapolated with the exact counts of the workload (64 + 64)."""
    from oracle import generate as G, llada, sampling as S
    cfg = llada.make_config(**{k: model_cfg[k] for k in ("d_model", "n_heads", "n_layers", "mlp_hidden_size", "vocab_size")},
                            max_sequence_length=model_cfg["max_sequence_length"])
    w = dict(synthetic_tensors(model_cfg, device, seed))
    model = llada.OracleModel(cfg, w)
    ids = lay["input_ids"].to(device).clone()
    NLd = NL
    total_len = lay["seq_len"] + lay["seq_len"] // lay["newline_every"]
    pos = torch.tensor([i for i in range(lay["image_start"], lay["image_start"] + total_len) if int(lay["input_ids"][0, i]) != NLd],
                       dtype=torch.long, device=device)
    noise = S.NoiseSource(torch.Generator(device=device).manual_seed(1), dtype=torch.bfloat16)
    unc_t, unc_i = lay["uncon_text"].to(device), lay["uncon_image"].to(device)

    def step(i, is_img):
        G._ti2ti_step(model, ids, i, is_img, 2, pos, noise, lay["text_start"], lay["text_end"], lay["seq_len"], GEN["text_steps"],
                      GEN["temperature"], GEN["text_temperature"], GEN["cfg_scale"], GEN["cfg_img"], unc_t, unc_i,
                      S.cosine_schedule, TEXT_VOCAB, CODEBOOK, True)

    def timed(n, is_img, first):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for j in range(n):
            step(first + j, is_img)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / n

    with torch.no_grad():
        step(0, False)
        step(32, True)
        t_text = timed(4, False, 1)
        t_img = timed(2, True, 33)
        # one bare forward, for s/forward and TFLOP/s
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(3):
            model(ids)
        torch.cuda.synchronize()
        t_fwd = (time.perf_counter() - t0) / 3
    per_sample = 64 * t_text + 64 * t_img
    d, ff, V, nl, L = cfg.d_model, cfg.mlp_hidden_size, cfg.vocab_size, cfg.n_layers, ids.shape[1]
    fwd_flops = nl * (2 * L * (4 * d * d + 3 * d * ff) + 4 * L * L * d) + 2 * L * d * V
    del model, w
    torch.cuda.empty_cache()
    return {"value": TOKENS_PER_SAMPLE / per_sample, "unit": "tokens/s", "kind": "oracle port of the reference loop, torch eager on cuda "
            "(cuBLAS + SDPA + ATen, full LM head, 192 forwards: the unused uncond_text forward is skipped, no .item() loops)",
            "sec_per_sample": per_sample, "sec_per_text_step": t_text, "sec_per_image_step": t_img, "sec_per_forward": t_fwd,
            "forward_tflops": fwd_flops / t_fwd / 1e12,
            "sample": "4 text-only steps + 2 image steps after 1 warm-up of each, extrapolated to 64 + 64"}


def run_reference_arm(args, rank: int):
    if rank != 0:
        return
    # interleave the weights over the NUMA nodes when numactl exists (a 2-socket host otherwise serves all threads from the
    # node that first touched the tensors); re-exec once under it
    import shutil
    if shutil.which("numactl") and not os.environ.get("MMDP_NUMACTL_DONE"):
        env = dict(os.environ, MMDP_NUMACTL_DONE="1")
        try:
            os.execvpe("numactl", ["numactl", "--interleave=all", sys.executable] + sys.argv, env)
        except OSError:
            pass
    cfg = MODEL_TINY if args.tiny else MODEL_8B
    vals = []
    r = None
    for _ in range(max(1, min(args.steps, 3))):  # each repetition = thread sweep x (1 warm-up + 3 timed) block forwards
        r = cpu_reference_sample(cfg)
        vals.append(r["tokens_per_s"])
    v = statistics.median(vals)
    out = {"impl": "reference", "metric": "denoised_tokens_per_sec", "value": v, "unit": "tokens/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * TOKENS_PER_SAMPLE / v, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
           "config": workload_config(args, 1),
           "cpu_baseline": {"value": v, "unit": "tokens/s", "cores": r["cores"], "kind": "port", "sample": r["sample"], "cpu": r["cpu"],
                            "thread_sweep_sec_per_block": r["thread_sweep_sec_per_block"], "repetitions_tokens_per_s": vals,
                            "numactl_interleave": bool(os.environ.get("MMDP_NUMACTL_DONE"))},
           "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "detail": {k: r[k] for k in ("t_block", "t_head_text", "t_head_img", "t_text_step", "t_image_step", "sec_per_sample")}}
    print(json.dumps(out), flush=True)


def workload_config(args, n_gpus):
    return {"workload": "MMaDA-Parallel-A 8B, 1 prompt per GPU, 512x512 (1024 VQ tokens) + 256 text tokens, timesteps=64, "
                        "text_steps=128, cfg_img=4.0, cfg_scale=0, temperature=1.0, text_temperature=0 (BASELINE configs[1]"
                        + ("; TINY MODEL - plumbing check only, not a valid number" if args.tiny else "") + ")",
            "seq_len": 2414, "forwards_per_sample": 192,
            "parallelism": (f"tensor-parallel x{n_gpus} (one prompt; heads/ff/vocab split, " + ("fused reduce+residual+norm+broadcast kernel over NVLink peer memory)" if getattr(args, "tp_collective", "p2p") == "p2p" else "fp32 all-reduce over NCCL)") if getattr(args, "tp", False) and n_gpus > 1
                            else f"replicas x{n_gpus} (independent prompts, no collective)"),
            "weights": "synthetic normal(0, 0.02) bf16, seeded", "l2": "16.2 GB of weights streamed per forward >> 126 MB L2 (no flush needed)"}


# ------------------------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------------------------
def model_namespace(model_cfg: dict):
    from types import SimpleNamespace
    return SimpleNamespace(**model_cfg, n_kv_heads=None, embedding_size=model_cfg["vocab_size"], rope_theta=500000.0,
                           rms_norm_eps=1e-5, rope=True, rope_full_precision=True, include_bias=False, weight_tying=False)


def synthetic_tensors(model_cfg: dict, device: str, seed: int):
    """Yields (HF name, bf16 tensor on `device`) of a seeded random-init model: normal(0, 0.02) matrices, unit norms."""
    g = torch.Generator(device=device).manual_seed(seed)
    d, ff, V = model_cfg["d_model"], model_cfg["mlp_hidden_size"], model_cfg["vocab_size"]

    def mk(*shape, ones=False):
        if ones:
            return torch.ones(shape, dtype=torch.bfloat16, device=device)
        return torch.empty(shape, dtype=torch.bfloat16, device=device).normal_(0.0, 0.02, generator=g)

    yield "model.transformer.wte.weight", mk(V, d)
    yield "model.transformer.ff_out.weight", mk(V, d)
    yield "model.transformer.ln_f.weight", mk(d, ones=True)
    for i in range(model_cfg["n_layers"]):
        p = f"model.transformer.blocks.{i}."
        for n in ("q_proj", "k_proj", "v_proj", "attn_out"):
            yield p + n + ".weight", mk(d, d)
        yield p + "ff_proj.weight", mk(ff, d)
        yield p + "up_proj.weight", mk(ff, d)
        yield p + "ff_out.weight", mk(d, ff)
        yield p + "attn_norm.weight", mk(d, ones=True)
        yield p + "ff_norm.weight", mk(d, ones=True)


def build_model(model_cfg: dict, device: str, seed: int):
    from mmada_parallel_b200.model import LLaDAForMultiModalGeneration
    m = LLaDAForMultiModalGeneration(model_namespace(model_cfg), max_seq_len=model_cfg["max_sequence_length"], max_batch=1, device=device)
    for name, t in synthetic_tensors(model_cfg, device, seed):
        assert m.set_weight(name, t)
    m.load_state_dict({}, strict=True)
    torch.cuda.synchronize()
    return m


def build_tp_model(model_cfg: dict, device: str, seed: int, rank: int, world: int, collective: str = "p2p"):
    """Tensor-parallel model (BASELINE config 4): every rank materialises the same seeded tensors and keeps its shard."""
    from mmada_parallel_b200.tensor_parallel import TensorParallelLLaDA
    sd = dict(synthetic_tensors(model_cfg, device, seed))
    m = TensorParallelLLaDA(model_namespace(model_cfg), sd, rank, world, max_seq_len=model_cfg["max_sequence_length"], device=device,
                            text_vocab_size=TEXT_VOCAB, codebook_size=CODEBOOK, collective=collective)
    del sd
    torch.cuda.empty_cache()
    torch.cuda.synchronize()
    return m


def algorithmic_flops_per_sample(c: dict, L: int = 2414):
    d, ff, V, nl = c["d_model"], c["mlp_hidden_size"], c["vocab_size"], c["n_layers"]
    body = nl * (2 * L * (4 * d * d + 3 * d * ff) + 4 * L * L * d)
    head_text, head_img = 2 * 256 * d * V, 2 * 1024 * d * CODEBOOK
    return 192 * body + 128 * head_text + 128 * head_img  # minimal-equivalent work (BASELINE.md section 3)


def measure_variant_m(args, rank: int, world: int, device: str, steps: int, warmup: int):
    """Variant M (BASELINE configs[4]: MMaDA-Parallel-M 8B, MagViT-v2 tokenizer ids, one prompt per GPU): L = 2341, B = 2
    (cond + uncond) on every one of the 128 steps, 64 image steps (SURVEY.md 8d synthetic input M). Public API call with host
    inputs = e2e. Returns the record on every rank (the time is the max over ranks)."""
    from types import SimpleNamespace
    from mmada_parallel_b200 import _lib
    from mmada_parallel_b200.mmada import MMadaModelLM
    from mmada_parallel_b200.parallel import max_over_ranks
    import torch.distributed as dist
    model_cfg = MODEL_TINY if args.tiny else MODEL_8B
    ns = model_namespace(model_cfg)
    ns.mask_token_id = MASK
    m = MMadaModelLM(ns, max_seq_len=model_cfg["max_sequence_length"], max_batch=2, device=device)
    for name, t in synthetic_tensors(model_cfg, device, 1000):
        assert m.set_weight(name, t)
    m.load_state_dict({}, strict=True)
    g = torch.Generator().manual_seed(rank)
    tvoc, soi, eoi, bos = 126349, 126085, 126086, 126080
    inp = torch.cat([torch.tensor([126340, soi]), torch.randint(tvoc, tvoc + CODEBOOK, (1024,), generator=g), torch.tensor([eoi]),
                     torch.randint(0, 126000, (32,), generator=g)])
    unc = inp.clone()
    unc[-32:] = torch.randint(0, 126000, (32,), generator=g)
    conf = SimpleNamespace(model=SimpleNamespace(mmada=SimpleNamespace(num_vq_tokens=1024, codebook_size=CODEBOOK)),
                           dataset=SimpleNamespace(preprocessing=SimpleNamespace(max_seq_length=256)))

    class Tok:
        bos_token_id = bos

        def __len__(self):
            return tvoc

    kw = dict(input_ids=inp, uncond_input_ids=unc, text_cfg=2.5, image_cfg=4.0, text_steps=128, image_steps=64,
              reserved_token_mapping={"<|soi|>": soi, "<|eoi|>": eoi}, config=conf, uni_prompting=SimpleNamespace(text_tokenizer=Tok()))
    rng = torch.Generator(device=device).manual_seed(42 + rank)
    L = inp.numel() + 1026 + 256
    with torch.no_grad():
        for _ in range(warmup):
            m.interleave_generate(generator=rng, **kw)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            img, txt = m.interleave_generate(generator=rng, **kw)
            txt.cpu()
        e1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = max_over_ranks(e0.elapsed_time(e1), device=device)
        # roofline of the dominant kernel on this workload (rank 0, one profiled sample)
        prof = None
        if rank == 0:
            _lib.lib.mmdp_prof_enable(1)
            m.interleave_generate(generator=rng, **kw)
            prof = _lib.prof_summary()
            _lib.lib.mmdp_prof_enable(0)
        if world > 1:
            dist.barrier()
    del m
    torch.cuda.empty_cache()
    v = world * steps * TOKENS_PER_SAMPLE / (ms / 1e3)
    c = model_cfg
    d, ff, V, nl = c["d_model"], c["mlp_hidden_size"], c["vocab_size"], c["n_layers"]
    flops = 128 * (2 * nl * (2 * L * (4 * d * d + 3 * d * ff) + 4 * L * L * d) + 2 * 2 * 256 * d * V) + 64 * 2 * 2 * 1024 * d * CODEBOOK
    rec = {"metric": "denoised_tokens_per_sec", "value": v, "unit": "tokens/s", "n_gpus": world, "steps": steps, "warmup": warmup,
           "ms_per_step": ms / steps, "scaling": "weak",
           "config": {"workload": "MMaDA-Parallel-M 8B (BASELINE configs[4] shape per GPU): 1 prompt per GPU, L=2341, CFG batch 2 on each of 128 "
                                  "steps, 64 image steps, text_cfg=2.5, image_cfg=4.0", "parallelism": f"replicas x{world} (no collective)",
                      "gemm_kernel": "cta_group::2 pair kernel (M = 4682: 19 pair m-tiles; the default for M > 256, MMDP_GEMM_PAIR=0 routes the 1-CTA kernel)"},
           "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": int(inp.numel() * 16), "d2h_bytes_per_step": 256 * 8},
           "algorithmic_pflop_per_sample": flops / 1e15,
           "whole_step_tflops_per_gpu": flops * steps / (ms / 1e3) / 1e12}
    if prof is not None:
        peaks = load_peaks()
        gm, gf, gn = prof["gemm"]
        rec["roofline"] = {"kernel": "gemm_pair_kernel / gemm_bf16_kernel (tcgen05, all epilogues)", "bound": "tensor", "achieved": gf / (gm / 1e3) / 1e12 if gm else None,
                           "peak": peaks[0], "unit": "TFLOP/s", "frac": (gf / (gm / 1e3) / 1e12 / peaks[0]) if gm else None, "peak_source": peaks[1],
                           "launches": gn, "avg_launch_ms": gm / max(1, gn)}
        rec["kernel_breakdown_one_sample_ms"] = {"gemm": gm, "attention": prof["attention"][0], "row_kernels": prof["row"][0], "sampling": prof["sampling"][0],
                                                 "attention_tflops": prof["attention"][1] / (prof["attention"][0] / 1e3) / 1e12 if prof["attention"][0] else None}
    return rec


def run_variant_m(args, rank, local_rank, world):
    import torch.distributed as dist
    device = f"cuda:{local_rank}"
    torch.cuda.set_device(device)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(device))
    rec = measure_variant_m(args, rank, world, device, args.steps, args.warmup)
    if rank == 0:
        rec.update({"higher_is_better": True, "vs_baseline": None, "dtype": "bf16", "data": "synthetic"})
        print(json.dumps(rec), flush=True)
    if world > 1:
        dist.destroy_process_group()


def load_peaks():
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return peaks.get("bf16_tflops_sustained", 1400.0), "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)", peaks
    except Exception:
        return 1400.0, "fallback ~1.4 PFLOP/s sustained (B200_PROFILING.md)", {}


def measure_vq_decode(device: str, iters: int = 10):
    """VQ decode reported separately (SURVEY 8d): MAGVITv2.decode_code, 1024 code ids -> 3 x 512 x 512 (full-size decoder,
    synthetic weights), through the public mirror; plus the TF32 conv engine's share from the live launch profile."""
    from mmada_parallel_b200 import _lib
    from mmada_parallel_b200.magvit import MAGVITv2
    m = MAGVITv2(max_batch=1, device=device)
    g = torch.Generator().manual_seed(0)
    sd = {}
    for name, shape in m.decoder.parameter_shapes().items():
        if len(shape) == 4:
            sd[name] = torch.randn(shape, generator=g) * (1.0 / (shape[1] * shape[2] * shape[3])) ** 0.5
        elif name.endswith("weight"):
            sd[name] = 1.0 + 0.1 * torch.randn(shape, generator=g)
        else:
            sd[name] = 0.05 * torch.randn(shape, generator=g)
    m.load_state_dict(sd)
    ids = torch.randint(0, CODEBOOK, (1, 1024), generator=g).to(device)
    for _ in range(3):
        m.decode_code(ids)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        out = m.decode_code(ids)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    _lib.lib.mmdp_prof_enable(1)
    m.decode_code(ids)
    prof = _lib.prof_summary()
    _lib.lib.mmdp_prof_enable(0)
    cm, cf, cn = prof["gemm"]
    rm, rb, rn = prof["row"]
    return {"ms_per_image": ms, "image": "1024 ids -> 3x512x512 fp32", "conv_tf32_ms": cm, "conv_tf32_launches": cn,
            "conv_tf32_tflops": cf / (cm / 1e3) / 1e12 if cm else None, "conv_flops_per_image": cf,
            "tf32_peak_nominal_tflops": 1100.0, "frac_of_nominal_tf32": (cf / (cm / 1e3) / 1e12 / 1100.0) if cm else None,
            "row_kernels_ms": rm, "row_kernels_GBps": rb / (rm / 1e3) / 1e9 if rm else None,
            "preview_path_cost_ms": 38 * ms, "note": "the step-wise preview loop (A/app.py) decodes after each of its 38 image steps"}


def measure_tensor_parallel(args, model_cfg, device, rank, world, replica_model, steps: int):
    """BASELINE configs[3]: ONE sample tensor-parallel over the `world` GPUs (strong scaling). Runs on every rank; includes a
    parity self-check the driver's multi-GPU lease can see: logits of the TP forward against the single-GPU forward of the
    same (seed-1000) weights, and the ranks' final ids compared."""
    import torch.distributed as dist
    from mmada_parallel_b200.generators.parallel_generator import DenoiseState, denoise_loop
    from mmada_parallel_b200.parallel import max_over_ranks
    from mmada_parallel_b200.schedule import cosine_schedule
    tp = build_tp_model(model_cfg, device, 1000, rank, world)
    lay = synthetic_layout(seed=0)
    ids = lay["input_ids"].to(device)
    text_rows = torch.arange(lay["text_start"], lay["text_end"], dtype=torch.int32, device=device)
    with torch.no_grad():
        from mmada_parallel_b200 import _lib
        a_tp, _ = tp.forward_rows(ids, rows_a=text_rows)
        a_1, _ = replica_model.forward_rows(ids, rows_a=text_rows)
        # yardstick: the same single-GPU forward with the other GEMM kernel (1-CTA tiles + split-K tail instead of CTA pairs) -
        # another valid accumulation order. A 32-layer random-weight network amplifies 1-ulp differences, so the bound for
        # the TP forward is "as close to the single-GPU forward as two single-GPU schedules are to each other" (x1.5);
        # the strict 4-ulp bound is enforced on the 2-layer model in tests/test_gpu_tp.py.
        _lib.lib.mmdp_set_gemm_pair(0)
        a_alt, _ = replica_model.forward_rows(ids, rows_a=text_rows)
        _lib.lib.mmdp_set_gemm_pair(1)
        scale = a_1.float().abs().max().item()
        err = (a_tp.float() - a_1.float()).abs()
        max_ulp = err.max().item() / (scale * 2.0 ** -8)
        mean_ulp = err.mean().item() / (scale * 2.0 ** -8)
        yard = (a_alt.float() - a_1.float()).abs()
        yard_max, yard_mean = yard.max().item() / (scale * 2.0 ** -8), yard.mean().item() / (scale * 2.0 ** -8)
        argmax_equal = float((a_tp.float().argmax(-1) == a_1.float().argmax(-1)).float().mean())
        argmax_yard = float((a_alt.float().argmax(-1) == a_1.float().argmax(-1)).float().mean())
        pos_args = {k: lay[k] for k in ("text_start", "text_end", "image_start", "seq_len", "newline_every")}
        loop_kw = dict(text_steps=GEN["text_steps"], timesteps=GEN["timesteps"], temperature=GEN["temperature"],
                       text_temperature=GEN["text_temperature"], cfg_scale=GEN["cfg_scale"], cfg_img=GEN["cfg_img"],
                       noise_schedule=cosine_schedule, text_vocab_size=TEXT_VOCAB, codebook_size=CODEBOOK)
        rng = torch.Generator(device=device).manual_seed(4242)  # identical on every rank: the ranks draw the same noise

        def new_state():
            return DenoiseState(tp, lay["input_ids"], uncon_text=lay["uncon_text"], uncon_image=lay["uncon_image"],
                                cfg_scale=GEN["cfg_scale"], cfg_img=GEN["cfg_img"], codebook_size=CODEBOOK, **pos_args)

        denoise_loop(new_state(), generator=rng, **loop_kw)  # warm-up sample
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        final = None
        for _ in range(steps):
            final = denoise_loop(new_state(), generator=rng, **loop_kw)
        e1.record()
        dist.barrier()
        torch.cuda.synchronize()
        ms = max_over_ranks(e0.elapsed_time(e1), device=device)
        # where the tensor-parallel sample spends its time (rank 0's launches bracketed by CUDA events; every rank runs the pass
        # because the forward contains the cross-rank flags). "row" = reduce + residual + norm + broadcast kernels incl. their
        # waits for the peers, "gemm" includes the fused reduce-scatter pushes.
        _lib.lib.mmdp_prof_enable(1)
        denoise_loop(new_state(), generator=rng, **loop_kw)
        tp_prof = _lib.prof_summary()
        _lib.lib.mmdp_prof_enable(0)
        dist.barrier()
        # ranks in lock-step: every rank's final id buffer equals rank 0's
        mine = final[0].clone()
        ref = mine.clone()
        dist.broadcast(ref, src=0)
        same = torch.tensor([1 if torch.equal(mine, ref) else 0], device=device)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        # the same model with the OTHER row-chunk schedule (1 chunk: collective traffic and GEMMs of a layer strictly alternate;
        # 2 chunks on two streams: one chunk's NVLink traffic under the other's GEMMs), one sample
        one_chunk_tok_s = None
        main_chunks = int(getattr(tp, "chunks", 1))
        if getattr(args, "tp_alt_schedule", False):  # opt-in: its numbers are on record (profiles/r02), the default run stays minimal
            tp.chunks, tp._ctx_key = (1 if main_chunks == 2 else 2), None
            dist.barrier()
            torch.cuda.synchronize()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            denoise_loop(new_state(), generator=rng, **loop_kw)
            c1.record()
            dist.barrier()
            torch.cuda.synchronize()
            one_chunk_tok_s = TOKENS_PER_SAMPLE / (max_over_ranks(c0.elapsed_time(c1), device=device) / 1e3)
    del tp
    torch.cuda.empty_cache()
    # the NCCL all-reduce formulation (round 1) on the same workload, one sample: what the peer-memory collective replaces
    nccl_tok_s = None
    try:
        tpn = build_tp_model(model_cfg, device, 1000, rank, world, collective="nccl")
        with torch.no_grad():
            def st_n():
                return DenoiseState(tpn, lay["input_ids"], uncon_text=lay["uncon_text"], uncon_image=lay["uncon_image"],
                                    cfg_scale=GEN["cfg_scale"], cfg_img=GEN["cfg_img"], codebook_size=CODEBOOK, **pos_args)
            dist.barrier()
            torch.cuda.synchronize()
            n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n0.record()
            denoise_loop(st_n(), generator=rng, **loop_kw)
            n1.record()
            dist.barrier()
            torch.cuda.synchronize()
            nccl_tok_s = TOKENS_PER_SAMPLE / (max_over_ranks(n0.elapsed_time(n1), device=device) / 1e3)
        del tpn
        torch.cuda.empty_cache()
    except Exception as e:
        nccl_tok_s = f"error: {type(e).__name__}: {e}"[:200]
    v = steps * TOKENS_PER_SAMPLE / (ms / 1e3)
    return {"metric": "denoised_tokens_per_sec", "value": v, "nccl_allreduce_baseline_tokens_per_s": nccl_tok_s,
            "row_chunks": main_chunks, "other_row_chunk_schedule": {"row_chunks": 1 if main_chunks == 2 else 2, "tokens_per_s": one_chunk_tok_s},
            "collective": "GEMM-fused reduce-scatter + reduce/residual/RMSNorm/broadcast kernel over NVLink peer memory (csrc/tp_collective.cu); "
                          "row_chunks = 2: two row chunks on two streams, one chunk's NVLink traffic under the other's GEMMs (default from TP=4)",
            "kernel_breakdown_one_sample_ms": {"gemm_incl_scatter_push": tp_prof["gemm"][0], "attention": tp_prof["attention"][0],
                                               "reduce_norm_broadcast_and_waits": tp_prof["row"][0], "sampling": tp_prof["sampling"][0]}, "unit": "tokens/s", "n_gpus": world, "steps": steps, "scaling": "strong",
            "ms_per_step": ms / steps, "config": {"workload": "BASELINE configs[3]: ONE prompt, tensor-parallel attention/MLP/LM head over the GPUs",
                                                  "parallelism": f"tensor-parallel x{world}"},
            "tp_parity": {"logits_max_err_bf16_ulp_of_scale": max_ulp, "logits_mean_err_bf16_ulp_of_scale": mean_ulp,
                          "yardstick_two_single_gpu_schedules_max_ulp": yard_max, "yardstick_mean_ulp": yard_mean,
                          "ok": bool(max_ulp <= max(4.0, 1.5 * yard_max) and mean_ulp <= max(0.25, 1.5 * yard_mean)),
                          "text_row_argmax_agreement": argmax_equal, "yardstick_argmax_agreement": argmax_yard,
                          "ranks_final_ids_identical": bool(int(same.item()) == 1),
                          "against": "single-GPU forward of the same 32-layer weights on this rank (256 text rows x V); yardstick = the same "
                                     "single-GPU forward with the 1-CTA GEMM kernel instead of the CTA-pair kernel"}}


DUMP_MAX_ELEMENTS = 1 << 22  # per array: 16 MB of float32


def dump_outputs(out_dir: str, st) -> None:
    """Writes what the last timed sample computed as `out_dir/<name>.npy`, for comparing two builds output for output:
    `ids` is the final id buffer denoise_loop returns (float64, exact for token ids); `text_logits` and `image_logits` are the
    buffers of the sample's last conditional forward (text rows x vocabulary, VQ rows x codebook), as float32. An array with
    more than DUMP_MAX_ELEMENTS elements is written as a fixed, seeded sample of its flattened elements (the same positions
    in every run)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("ids", st.ids.double()), ("text_logits", st.text_logits.float()), ("image_logits", st.cond_vq.float())):
        flat = t.reshape(-1)
        if flat.numel() > DUMP_MAX_ELEMENTS:
            keep = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ELEMENTS].sort().values
            t = flat[keep.to(flat.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2, help="timed samples")
    ap.add_argument("--warmup", type=int, default=3, help="untimed samples before them")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed samples, write what the last one computed as DIR/<name>.npy "
                    "(rank 0)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--tiny", action="store_true", help="2-layer d=256 model: plumbing check only (INVALID as a benchmark number)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the sub-records (tensor-parallel at N > 1, variant M, torch-eager GPU "
                    "baseline, VQ decode timing)")
    ap.add_argument("--variant", default="a", choices=["a", "m"], help="a = BASELINE configs[1] (the contract metric); m = extra line for "
                    "variant M (interleave_generate, CFG batch 2 every step, BASELINE configs[4] per GPU)")
    ap.add_argument("--tp-alt-schedule", action="store_true", help="tp record: also time one sample with the other row-chunk schedule "
                    "(two chunks on two streams instead of one)")
    ap.add_argument("--tp-collective", default="p2p", choices=["p2p", "nccl"], help="--tp: fused reduce + residual + norm + broadcast over "
                    "NVLink peer memory (default) or the NCCL all-reduce baseline")
    ap.add_argument("--tp", action="store_true", help="N > 1: ONE sample tensor-parallel over the N GPUs (strong scaling, NCCL "
                    "all-reduce) instead of N independent replicas")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl != "b200" or args.variant != "a"):
        ap.error("--dump-outputs writes the outputs of the variant A path of --impl b200")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if args.variant == "m":
        run_variant_m(args, rank, local_rank, world)
        return

    import torch.distributed as dist
    from mmada_parallel_b200 import _lib
    from mmada_parallel_b200.generators.parallel_generator import DenoiseState, denoise_loop, generate_ti2ti
    from mmada_parallel_b200.parallel import max_over_ranks
    from mmada_parallel_b200.schedule import cosine_schedule

    device = f"cuda:{local_rank}"
    torch.cuda.set_device(device)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(device))
    model_cfg = MODEL_TINY if args.tiny else MODEL_8B
    tp_mode = args.tp and world > 1
    if tp_mode:
        model = build_tp_model(model_cfg, device, 1000, rank, world, collective=args.tp_collective)
        lay = synthetic_layout(seed=0)  # ONE prompt, all ranks work on it
    else:
        model = build_model(model_cfg, device, seed=1000)
        lay = synthetic_layout(seed=rank)  # every rank denoises its own prompt
    host_ids = lay["input_ids"].pin_memory()
    pos_args = {k: lay[k] for k in ("text_start", "text_end", "image_start", "seq_len", "newline_every")}
    gen = GEN
    loop_kw = dict(text_steps=gen["text_steps"], timesteps=gen["timesteps"], temperature=gen["temperature"],
                   text_temperature=gen["text_temperature"], cfg_scale=gen["cfg_scale"], cfg_img=gen["cfg_img"],
                   noise_schedule=cosine_schedule, text_vocab_size=TEXT_VOCAB, codebook_size=CODEBOOK)

    def new_state():
        return DenoiseState(model, lay["input_ids"], uncon_text=lay["uncon_text"], uncon_image=lay["uncon_image"],
                            cfg_scale=gen["cfg_scale"], cfg_img=gen["cfg_img"], codebook_size=CODEBOOK, **pos_args)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    rng = torch.Generator(device=device).manual_seed(42 if tp_mode else 42 + rank)  # TP ranks must draw identical noise
    with torch.no_grad():
        for _ in range(args.warmup):
            denoise_loop(new_state(), generator=rng, **loop_kw)
        # ---- timed region 1: inputs resident in HBM ("value")
        states = [new_state() for _ in range(args.steps)]
        clocks = ClockSampler(local_rank)
        barrier()
        if rank == 0:
            clocks.start()
        _lib.lib.mmdp_launch_count(1)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for st in states:
            denoise_loop(st, generator=rng, **loop_kw)
        ev1.record()
        barrier()
        launches = int(_lib.lib.mmdp_launch_count(0))
        clock_info = clocks.stop() if rank == 0 else None
        ms_value = max_over_ranks(ev0.elapsed_time(ev1), device=device)

        # ---- timed region 2: through the public API with HOST buffers ("e2e"): H2D of the inputs + D2H of the result inside
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        with quiet():
            for _ in range(args.steps):
                img, txt = generate_ti2ti(model, host_ids, uncon_text=lay["uncon_text"], uncon_image=lay["uncon_image"], generator=rng,
                                          text_gen_length=gen["text_gen_length"], text_block_length=gen["text_block_length"],
                                          **pos_args, **{k: v for k, v in loop_kw.items()})
        e1.record()
        barrier()
        ms_e2e = max_over_ranks(e0.elapsed_time(e1), device=device)
        h2d = states[0].bytes_h2d()
        d2h = host_ids.numel() * 8

        # ---- roofline pass (rank 0): one sample with every launch bracketed by CUDA events
        prof = None
        if rank == 0 or tp_mode:  # tensor-parallel: every rank must take part (the forward contains collectives)
            _lib.lib.mmdp_prof_enable(1)
            denoise_loop(new_state(), generator=rng, **loop_kw)
            prof = _lib.prof_summary()
            _lib.lib.mmdp_prof_enable(0)
        barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, states[-1])

    # ---- sub-records on the other BASELINE configs (every rank takes part where a collective or a barrier is involved)
    extras = {}
    states = st = None  # (they hold the model and ~120 MB of device buffers each)
    if not tp_mode and not args.no_extras:
        if world > 1:
            try:
                extras["tp"] = measure_tensor_parallel(args, model_cfg, device, rank, world, model, steps=max(1, min(args.steps, 3)))
            except Exception as e:  # a failing sub-record must not take the contract line down; it is reported instead
                extras["tp"] = {"error": f"{type(e).__name__}: {e}"[:400]}
                dist.barrier()
        del model
        torch.cuda.empty_cache()
        try:
            extras["variant_m"] = measure_variant_m(args, rank, world, device, steps=max(1, min(args.steps, 2)), warmup=1)
        except Exception as e:
            extras["variant_m"] = {"error": f"{type(e).__name__}: {e}"[:400]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    n_samples = args.steps if tp_mode else world * args.steps
    total_tokens = n_samples * TOKENS_PER_SAMPLE
    value = total_tokens / (ms_value / 1e3)
    e2e_value = total_tokens / (ms_e2e / 1e3)
    peak_tf, peak_src, peaks = load_peaks()
    gemm_ms, gemm_flops, gemm_n = prof["gemm"]
    att_ms, att_flops, att_n = prof["attention"]
    row_ms, row_bytes, row_n = prof["row"]
    smp_ms, smp_bytes, smp_n = prof["sampling"]
    achieved = gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms else 0.0
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json"))).get("gemm_dram_bytes_per_launch")
    except Exception:
        pass
    flops_sample = algorithmic_flops_per_sample(model_cfg)
    hbm = peaks.get("hbm_gbs", 6650.0)
    out = {
        "metric": "denoised_tokens_per_sec", "value": value, "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_value / args.steps, "higher_is_better": True,
        "scaling": "strong" if tp_mode else "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(args, world),
        "e2e": {"value": e2e_value, "unit": "tokens/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches,
        "clocks": clock_info,
        "roofline": {"kernel": "gemm_pair_kernel / gemm_bf16_kernel (tcgen05 cta_group::2 / ::1, all epilogues)", "bound": "tensor", "achieved": achieved, "peak": peak_tf,
                     "unit": "TFLOP/s", "frac": achieved / peak_tf if peak_tf else None, "traffic": traffic,
                     "peak_source": peak_src, "launches": gemm_n, "avg_launch_ms": gemm_ms / max(1, gemm_n),
                     "algorithmic_flops_per_launch": gemm_flops / max(1, gemm_n)},
        "kernel_breakdown_one_sample_ms": {"gemm": gemm_ms, "attention": att_ms, "row_kernels": row_ms, "sampling": smp_ms,
                                           "attention_tflops": att_flops / (att_ms / 1e3) / 1e12 if att_ms else None,
                                           "row_GBps": row_bytes / (row_ms / 1e3) / 1e9 if row_ms else None,
                                           "sampling_GBps": smp_bytes / (smp_ms / 1e3) / 1e9 if smp_ms else None,
                                           "sampling_frac_of_hbm_peak": (smp_bytes / (smp_ms / 1e3) / 1e9 / hbm) if smp_ms else None,
                                           "note": "per-launch CUDA events serialise the launches: programmatic dependent launch overlap is "
                                                   "not visible here, the timed regions above include it"},
        # executed tensor work of one sample = the flops of the GEMM and attention launches actually made (profiled sample). It is
        # below BASELINE.md's "minimal-equivalent" 7.101 PFLOP: the last block computes its attention output / MLP only for the
        # rows whose logits are read (row window, output-invariant), 0.11 PFLOP per sample less.
        "executed_pflop_per_sample": (gemm_flops + att_flops) / 1e15,
        "baseline_minimal_pflop_per_sample": flops_sample / 1e15,
        "whole_step_tflops_executed_work": (gemm_flops + att_flops) * n_samples / (ms_value / 1e3) / 1e12,
        "whole_step_frac_of_peak": (gemm_flops + att_flops) * n_samples / (ms_value / 1e3) / 1e12 / (peak_tf * world),  # per-GPU fraction
    }
    out.update(extras)
    if world == 1 and not tp_mode:
        if not args.no_cpu_baseline:
            r = cpu_reference_sample(model_cfg)
            out["cpu_baseline"] = {"value": r["tokens_per_s"], "unit": "tokens/s", "cores": r["cores"], "kind": "port",
                                   "sample": r["sample"], "sec_per_sample": r["sec_per_sample"], "cpu": r["cpu"],
                                   "thread_sweep_sec_per_block": r["thread_sweep_sec_per_block"]}
        else:
            out["cpu_baseline"] = None
        if not args.no_extras:
            try:
                g = gpu_eager_baseline(model_cfg, device, lay)
                g["speedup_e2e_over_eager"] = e2e_value / g["value"]
                out["gpu_eager_baseline"] = g
            except Exception as e:
                out["gpu_eager_baseline"] = {"error": f"{type(e).__name__}: {e}"[:400]}
            try:
                out["vq_decode"] = measure_vq_decode(device)
            except Exception as e:
                out["vq_decode"] = {"error": f"{type(e).__name__}: {e}"[:400]}
    else:
        out["cpu_baseline"] = None
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
