#!/usr/bin/env python
"""Benchmark of the hot path: tokens/sec of the Llama-2-7B LoRA (r=16, q_proj,v_proj) SFT step, seq 2048,
batch 8 per GPU, bf16, synthetic instruction pairs, random-init weights (BASELINE.json configs[1]).

  python bench.py --gpus N --steps K --warmup W            native arm (libdtxtune.so, one process per GPU)
  python bench.py --impl reference --gpus N ...             CPU arm: the oracle restatement of the reference step
                                                            on the host cores (the reference itself cannot run here)

A "step" = forward + backward + (NCCL all-reduce) + clip + AdamW on one batch of 8 x 2048 tokens per GPU.
`value`  : device-resident batches (dtx_step_device), wall clock over K steps between barriers, max over ranks.
`e2e`    : the same K steps through the public host API (pinned host int32 batches in, loss/grad-norm out).
`roofline`: the kernel with the largest share of the step - the CTA-pair tcgen05 GEMM with an MN-major B operand
            (`gemm2_kernel<1,0>`, 31.8 % of the step: the backward dX GEMMs) - timed alone with CUDA events at its largest
            per-layer shape (dh2 = d[gate|up] . [Wg;Wu]: 16384 x 4096 x 22016) against MEASURED_PEAKS.json's burst bf16 figure;
            `roofline_kernels` lists the same measurement for the other GEMM variants the step runs (SwiGLU-forward epilogue
            at the gate|up shape, SwiGLU-backward epilogue); `step_roofline` is the whole step against the sustained figure
            with the algorithmic 28.36 GFLOP/token of BASELINE.md.
`ranks`  : per-rank device time per step (min / median / max), its forward+backward / all-reduce / optimizer split
            (CUDA events inside libdtxtune) and the rank's median SM clock during the timed region - what explains the
            1 -> N curve (the step is lock-step: the slowest GPU's clock sets the pace).
`--config 7b_varlen`: the same model on a length-distributed synthetic set (rows padded to the longest of their batch like
            DataCollatorForSeq2Seq, true row lengths passed to the step, which runs the batch packed - DESIGN.md 2.2): reports
            real (unpadded) tokens/s, `packed_steps`, `length_groups_per_step`.  DTX_VARLEN_SPLIT=0 / DTX_VARLEN_PACK=0: one pass
            at the padded shape / length groups, for A/B runs.
Other configs (not the headline metric): mistral7b_qlora (BASELINE configs[2]), 13b_full (configs[3], 8 GPUs), small_full, tiny.
`--dump-outputs DIR`: loss, grad-norm, lr of the last timed device-resident step and the trainable parameters after it, as .npy
            (seeded inputs and weights: the same arguments give the same inputs, so two builds compare array for array).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_TOKEN = 28.36e9  # BASELINE.md §2 (fwd GEMM + bwd dX GEMM + causal attention fwd/bwd + LoRA; no recompute)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"burst": d.get("bf16_tflops", 1590.0), "sustained": d.get("bf16_tflops_sustained", 1400.0),
                "hbm": d.get("hbm_gbs", 6650.0), "src": "MEASURED_PEAKS.json"}
    return {"burst": 1590.0, "sustained": 1400.0, "hbm": 6650.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in self.rows if len(r) >= 7 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "power_w": float(np.median(pw)) if pw else None}


class EnergyMeter:
    """NVML total-energy counter of one GPU (mJ since driver load): joules spent inside a timed region."""

    def __init__(self, index: int):
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            pynvml.nvmlDeviceGetTotalEnergyConsumption(self.h)
        except Exception:
            self.h = None

    def read_j(self):
        if self.h is None:
            return None
        try:
            return self.nv.nvmlDeviceGetTotalEnergyConsumption(self.h) / 1000.0
        except Exception:
            return None


def cpu_info():
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
        ram_gb = psutil.virtual_memory().available / 2**30
    except Exception:
        physical, ram_gb = logical, None
    return {"cpu_model": model, "logical_cpus": logical, "physical_cores": physical, "available_ram_gb": ram_gb}


def cpu_threads(info) -> int:
    """Deterministic torch thread count of the CPU arms.  On the 128-thread hosts of the GPU boxes torch's fp32 GEMM of this
    step is an order of magnitude SLOWER with every hardware thread than with a moderate count (r01: 4.3 vs 40 tokens/s);
    32 threads (or all physical cores on a smaller host) is what the round-1 calibration runs settled on."""
    return max(1, min(32, info["physical_cores"]))


def oracle_full_model_step(n_layers: int, seq_len: int, threads: int, warmup: int, steps: int):
    """Time the oracle (fp32 CPU restatement of the reference training step) on the FULL Llama-2-7B architecture: one sequence of
    `seq_len` tokens per step - forward, CE, backward, clip, AdamW through all `n_layers` decoder layers, embedding and lm_head.
    No extrapolation: every reported step is a measured whole-model step.  Weights are distinct fp32 tensors cut from a
    N(0, 0.02) pool (a fresh torch.randn of 6.7 G values would take minutes and is not part of the step)."""
    import torch
    from oracle import llama_lora as O
    torch.set_num_threads(threads)
    cfg = O.OracleConfig.llama2_7b(lora_r=16, lora_alpha=32.0, lr=1e-4, total_steps=100)
    cfg.n_layers = n_layers
    d, F, V = cfg.hidden, cfg.ffn, cfg.vocab
    t0 = time.perf_counter()
    pool = torch.randn(1 << 27, generator=torch.Generator().manual_seed(1)) * 0.02
    count = [0]

    def cut(*shape):
        n = int(np.prod(shape))
        count[0] += 1
        off = (count[0] * 1_000_003) % (pool.numel() - n + 1)
        return pool[off:off + n].view(*shape).clone()

    w = {"model.embed_tokens.weight": cut(V, d), "lm_head.weight": cut(V, d), "model.norm.weight": torch.ones(d)}
    for l in range(n_layers):
        p = f"model.layers.{l}."
        for n, shp in (("self_attn.q_proj", (d, d)), ("self_attn.k_proj", (d, d)), ("self_attn.v_proj", (d, d)),
                       ("self_attn.o_proj", (d, d)), ("mlp.gate_proj", (F, d)), ("mlp.up_proj", (F, d)), ("mlp.down_proj", (d, F))):
            w[p + n + ".weight"] = cut(*shp)
        w[p + "input_layernorm.weight"] = torch.ones(d)
        w[p + "post_attention_layernorm.weight"] = torch.ones(d)
    del pool
    tr = O.OracleTrainer(cfg, w, O.init_lora(cfg, 4321))
    t_init = time.perf_counter() - t0
    ts, losses = [], []
    for s in range(warmup + steps):
        batch = O.synthetic_batch(s, 0, 1, seq_len, V)
        t0 = time.perf_counter()
        log = tr.step([batch])
        if s >= warmup:
            ts.append(time.perf_counter() - t0)
            losses.append(log.loss)
    return {"sec_per_step": float(np.mean(ts)), "sec_steps": ts, "sec_init": t_init, "losses": losses, "layers": n_layers,
            "seq_len": seq_len, "warmup": warmup, "steps": steps}


def cpu_arm(warmup: int, steps: int):
    """Shared by `--impl reference` and the native arm's `cpu_baseline` leg."""
    info = cpu_info()
    threads = cpu_threads(info)
    layers, note = 32, None
    # fp32 weights 26.9 GB + ~1.1 GB of saved activations per layer for one 2048-token sequence
    need_gb = 27.0 + 32 * 1.2 + 6.0
    if info["available_ram_gb"] is not None and info["available_ram_gb"] < need_gb:
        layers = max(1, int((info["available_ram_gb"] - 8.0) / (27.0 / 32 + 1.2)))
        layers = min(32, layers)
        note = f"host has {info['available_ram_gb']:.0f} GB of free RAM: only {layers} of 32 layers fit (NOT the full model)"
    r = oracle_full_model_step(layers, 2048, threads, warmup, steps)
    v = 2048.0 / r["sec_per_step"]
    sample = (f"oracle (fp32 torch CPU restatement of cmd/tuning/train.py:196-299; the reference worker itself needs ray/peft/"
              f"deepspeed/CUDA and cannot run): full Llama-2-7B architecture ({layers} decoder layers + embedding + lm_head + CE), "
              f"LoRA r=16 q,v, one 2048-token sequence per step, fwd+bwd+clip+AdamW, {warmup} warm-up + {steps} timed steps, "
              f"every step measured (no extrapolation)")
    return {"value": v, "unit": "tokens/s", "cores": threads, "kind": "port", "sample": sample, "detail": r, "host": info,
            "torch_threads": threads, "same_model": layers == 32, "note": note}


def run_reference(args, rank: int):
    if rank != 0:
        return
    t0 = time.perf_counter()
    steps = max(1, min(args.steps, 2))  # a whole-model CPU step takes about a minute: 1 warm-up + 2 timed steps stay within minutes
    cb = cpu_arm(warmup=1, steps=steps)
    wall = time.perf_counter() - t0
    v = cb["value"]
    line = {"impl": "reference", "metric": "tokens/sec Llama-2-7B LoRA SFT seq2048", "value": v, "unit": "tokens/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": 1, "steps_requested": args.steps, "warmup_requested": args.warmup,
            "ms_per_step": 1000.0 * cb["detail"]["sec_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "Llama-2-7B LoRA r=16 q_proj,v_proj, seq 2048 (CPU arm: batch 1 sequence per step - a bounded sample "
                                   "of the 8-sequence GPU batch, same model, same sequence length)"},
            "cpu_baseline": dict(cb, wall_s=wall),
            "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# dram__bytes_read.sum + dram__bytes_write.sum of one launch of the profiled GEMMs at the bench shapes (ncu --set full):
# profiles/r01_ncu_dominant_gemm_final.txt (gate|up NT shape, plain epilogue), profiles/r02_ncu_gemm.txt (the backward variants:
# dX of gate|up with K = 22016 re-reads its operands 5.6x from DRAM at 99.5 % tensor activity - DESIGN.md 4.1 on why that
# costs neither time nor measurable energy).
GEMM_DRAM_BYTES = {"nt_gate_up": 2.0769e9, "nn_dh2": 5.2065e9, "nn_swiglu_bwd": 2.8669e9}


def time_step_gemms(torch, L):
    """CUDA-event timing of the CTA-pair tcgen05 GEMM variants the step actually launches, at their largest per-layer shapes."""
    import ctypes as C
    lib = L.load()
    M, d, F = 16384, 4096, 11008
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rnd = lambda *s, sc=0.05: (torch.randn(*s, device="cuda") * sc).to(torch.bfloat16)
    P = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    out = {}

    def timed(fn, flop, iters=10, idle_s=0.5, warm=3):
        # every leg starts from the same power state: after the 1 kW step the clocks take tens of milliseconds to settle, and
        # back-to-back legs measured 0.74 .. 0.95 of the burst peak for the same kernel depending on their order
        # (profiles/r02_bench_default_*.json before this pause).  idle_s = 0 + a long warm-up gives the power-capped figure.
        torch.cuda.synchronize()
        time.sleep(idle_s)
        for _ in range(warm):
            fn()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        s.record()
        for _ in range(iters):  # operands + output of every variant are >= 0.45 GB >> 126 MB L2: each launch streams from HBM
            fn()
        e.record()
        torch.cuda.synchronize()
        ms = s.elapsed_time(e) / iters
        return {"ms": ms, "tflops": flop / ms / 1e9}

    # (1) backward dX through the MLP up/gate weights: dh2[M, d] = dgu[M, 2F] . Wgu[2F, d]   (gemm2_kernel<B_MN=1, EPI_BF16>)
    dgu, wgu, dh = rnd(M, 2 * F), rnd(2 * F, d, sc=0.02), torch.empty(M, d, dtype=torch.bfloat16, device="cuda")
    out["nn_dh2"] = dict(timed(lambda: L.check(lib.dtx_gemm_bf16(P(dgu), 2 * F, 0, P(wgu), d, 1, None, 0, None, 0, 0, P(dh), d, None, 0,
                                                                 M, d, 2 * F, 0, 1, 0, stream)), 2.0 * M * d * 2 * F),
                         kernel="gemm2_kernel<B_MN=1, EPI_BF16>", shape_mnk=[M, d, 2 * F], alg_bytes=2.0 * (M * 2 * F + 2 * F * d + M * d))
    sus = timed(lambda: L.check(lib.dtx_gemm_bf16(P(dgu), 2 * F, 0, P(wgu), d, 1, None, 0, None, 0, 0, P(dh), d, None, 0,
                                                  M, d, 2 * F, 0, 1, 0, stream)), 2.0 * M * d * 2 * F, iters=100, idle_s=0.0, warm=100)
    out["nn_dh2"].update(ms_sustained=sus["ms"], tflops_sustained=sus["tflops"])  # 0.2 s warm-up + 0.2 s timed under the power cap
    # (2) forward gate|up projection with the SwiGLU epilogue: gu[M, 2F], act[M, F]   (gemm2_kernel<0, EPI_SWIGLU_FWD>)
    h2, gu, act = rnd(M, d), dgu, torch.empty(M, F, dtype=torch.bfloat16, device="cuda")
    out["nt_gate_up_swiglu"] = dict(timed(lambda: L.check(lib.dtx_gemm_fused(P(h2), d, P(wgu), d, 0, None, 0, None, 0, 0, P(gu), 2 * F, P(act), F,
                                                                             None, 0, 0, M, 2 * F, d, L.EPI_SWIGLU_FWD, stream)), 2.0 * M * 2 * F * d),
                                    kernel="gemm2_kernel<0, EPI_SWIGLU_FWD>", shape_mnk=[M, 2 * F, d],
                                    alg_bytes=2.0 * (M * d + 2 * F * d + M * 2 * F + M * F))
    # (3) backward through Wdown with the SwiGLU-backward epilogue: dgu[M, 2F] from dx[M, d] . Wdown[d, F] and saved gu
    dx, wdown, dgu2 = rnd(M, d), rnd(d, F, sc=0.02), torch.empty(M, 2 * F, dtype=torch.bfloat16, device="cuda")
    out["nn_swiglu_bwd"] = dict(timed(lambda: L.check(lib.dtx_gemm_fused(P(dx), d, P(wdown), F, 1, None, 0, None, 0, 0, P(dgu2), 2 * F, P(gu), 2 * F,
                                                                         None, 0, 0, M, F, d, L.EPI_SWIGLU_BWD, stream)), 2.0 * M * F * d),
                                kernel="gemm2_kernel<1, EPI_SWIGLU_BWD>", shape_mnk=[M, F, d],
                                alg_bytes=2.0 * (M * d + d * F + 2 * M * 2 * F))
    # (4) the plain NT kernel at the gate|up shape (r01's roofline leg, kept for continuity)
    out["nt_gate_up"] = dict(timed(lambda: L.check(lib.dtx_gemm_bf16(P(h2), d, 0, P(wgu), d, 0, None, 0, None, 0, 0, P(gu), 2 * F, None, 0,
                                                                     M, 2 * F, d, 0, 1, 0, stream)), 2.0 * M * 2 * F * d),
                             kernel="gemm2_kernel<0, EPI_BF16>", shape_mnk=[M, 2 * F, d], alg_bytes=2.0 * (M * d + 2 * F * d + M * 2 * F))
    del dgu, wgu, dh, h2, act, dx, wdown, dgu2
    torch.cuda.empty_cache()
    return out


def varlen_lengths(step: int, rank: int, batch: int, seq_len: int) -> np.ndarray:
    """Row lengths of the length-distributed synthetic set: instruction pairs are short-tailed in practice - a log-normal
    around a quarter of the cutoff, clipped to [16, seq_len]."""
    rng = np.random.default_rng(777 + rank * 1_000_003 + step)
    return np.clip(np.exp(rng.normal(np.log(seq_len / 4.0), 0.6, size=batch)), 16, seq_len).astype(np.int32)


DUMP_BYTES = 64 << 20  # what --dump-outputs may write in all


def dump_outputs(tr, out_dir: str, last_step, full: bool) -> None:
    """--dump-outputs: what the last device-resident timed step handed back - loss, grad-norm and learning rate - and the
    trainable parameters it left behind, one DIR/<checkpoint name>.npy each: the PEFT adapters (fp32) or, for a full fine-tune,
    the bf16 weights widened to fp32.  When the parameters exceed the budget, every tensor is cut to the same fraction of its
    elements at positions drawn from a fixed per-tensor seed (flattened, in index order)."""
    os.makedirs(out_dir, exist_ok=True)
    loss, gnorm, lr, _ = last_step
    arrays = {"loss": np.float32([loss]), "grad_norm": np.float32([gnorm]), "lr": np.float32([lr])}
    params = tr.export_weights() if full else tr.export_adapter()
    frac = min(1.0, (DUMP_BYTES - (1 << 20)) / (4.0 * sum(a.size for a in params.values())))  # 1 MB left for headers, scalars
    for i, (name, a) in enumerate(params.items()):
        if frac < 1.0:
            idx = np.sort(np.random.default_rng(i).choice(a.size, size=max(1, int(a.size * frac)), replace=False))
            a = a.reshape(-1)[idx]
        arrays[name] = (a.astype(np.uint32) << 16).view(np.float32) if full else a
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_native(args, rank: int, local_rank: int, world: int):
    import torch  # device memory for the resident batches, gloo rendezvous and the clock; no torch compute
    from datatunerx_b200 import lib as L
    from datatunerx_b200.tuning.data import batch_seq_len
    from datatunerx_b200.tuning.synthetic import synthetic_batch

    from datatunerx_b200.dist import Rendezvous
    rv = Rendezvous()
    torch.cuda.set_device(local_rank)

    lora_r, quant, varlen, full = 16, None, False, False
    if args.config == "13b_full":  # BASELINE.json configs[3]: Llama-2-13B full-parameter SFT bf16, seq 2048, data-parallel (beyond the reference)
        mc = L.ModelConfig(vocab=32000, hidden=5120, n_layers=40, n_heads=40, ffn=13824)
        B, S, full = 4, 2048, True
    elif args.config == "small_full":  # the same path at a size that fits one GPU with its whole optimizer state
        mc = L.ModelConfig(vocab=32000, hidden=2048, n_layers=8, n_heads=16, ffn=5504)
        B, S, full = 8, 2048, True
    elif args.config in ("7b", "7b_varlen"):
        mc = L.ModelConfig.llama2_7b()
        B, S = 8, 2048
        varlen = args.config == "7b_varlen"
    elif args.config == "mistral7b_qlora":  # BASELINE.json configs[2]: Mistral-7B QLoRA nf4 r=32, seq 4096 (not the headline metric)
        mc = L.ModelConfig(vocab=32000, hidden=4096, n_layers=32, n_heads=32, n_kv_heads=8, ffn=14336, max_seq=32768, sliding_window=4096)
        B, S, lora_r, quant = 4, 4096, 32, "int4"
    else:
        mc = L.ModelConfig(vocab=2048, hidden=256, n_layers=2, n_heads=2, ffn=768)
        B, S = 2, 256
    total = args.warmup + 2 * args.steps + 2
    tc = L.TrainConfig(micro_batch=B, seq_len=S, total_steps=max(total, 100), lora_r=lora_r, lora_alpha=32.0, lora_dropout=0.0, lr=1e-4 if not full else 1e-5,
                       full_finetune=full)
    nccl_id = rv.broadcast_bytes(L.nccl_unique_id)
    if os.environ.get("DTX_FWD_EXP_FMA"):  # A/B of the forward softmax's FMA-pipe exp2 fraction
        L.set_option("attn_fwd_exp_fma_every", int(os.environ["DTX_FWD_EXP_FMA"]))
    if os.environ.get("DTX_NF4_PREFETCH"):  # A/B of the side-stream NF4 expansion
        L.set_option("nf4_prefetch", int(os.environ["DTX_NF4_PREFETCH"]))
    if os.environ.get("DTX_VARLEN_SPLIT"):  # A/B of the length-group execution of ragged micro-batches
        L.set_option("varlen_split", int(os.environ["DTX_VARLEN_SPLIT"]))
    if os.environ.get("DTX_VARLEN_PACK"):  # A/B: packed single pass (default) vs length groups
        L.set_option("varlen_pack", int(os.environ["DTX_VARLEN_PACK"]))
    if os.environ.get("DTX_VARLEN_GROUP_COST"):
        L.set_option("varlen_group_cost", int(os.environ["DTX_VARLEN_GROUP_COST"]))
    if os.environ.get("DTX_GROUP_M"):  # rasterisation sweep of the CTA-pair GEMM (tools/gpu_round.sh sweep_gm)
        L.set_option("gemm_group_m", int(os.environ["DTX_GROUP_M"]))
    tr = L.Trainer(mc, tc, device=local_rank, rank=rank, world=world, nccl_id=nccl_id)
    tr.init_random_weights(1234)
    if quant:
        tr.quantize_base(quant)
    base_bytes = tr.base_weight_bytes
    if not full:
        tr.init_lora(4321)

    n_batches = 4
    host, lens_host = [], []
    for i in range(n_batches):
        ids, lab = synthetic_batch(i, rank, B, S, mc.vocab)
        if varlen:
            lens = varlen_lengths(i, rank, B, S)
            cur = batch_seq_len(lens.tolist(), S)
            for b in range(B):
                ids[b, lens[b]:] = 0
                lab[b, lens[b]:] = -100
                lab[b, :max(1, int(lens[b]) // 3)] = -100
            ids, lab = np.ascontiguousarray(ids[:, :cur]), np.ascontiguousarray(lab[:, :cur])
        else:
            lens, cur = np.full(B, S, dtype=np.int32), S
        host.append((ids, lab))
        lens_host.append((lens, cur))
    pinned = [(torch.from_numpy(a).pin_memory(), torch.from_numpy(b).pin_memory(), torch.from_numpy(l).pin_memory())
              for (a, b), (l, _) in zip(host, lens_host)]
    dev = [(a.cuda(non_blocking=False), b.cuda(non_blocking=False), l.cuda(non_blocking=False)) for a, b, l in pinned]
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        rv.barrier()

    def run(i, on_device):
        a, b, l = (dev if on_device else pinned)[i % n_batches]
        cur = lens_host[i % n_batches][1]
        return tr.step_ptr(a.data_ptr(), b.data_ptr(), on_device=on_device, seq_lens_ptr=l.data_ptr() if varlen else 0,
                           seq_len_batch=cur)

    losses = [run(i, True)[0] for i in range(args.warmup)]

    sampler = ClockSampler(local_rank)
    sampler.start()
    meter = EnergyMeter(local_rank)
    # ---- timed region 1: device-resident inputs ----
    launches0 = tr.launch_count
    barrier()
    e0 = meter.read_j()
    t0 = time.perf_counter()
    dev_ms, segs, groups = [], [], []
    real_tokens = padded_tokens = 0
    for i in range(args.steps):
        last = run(i, True)
        losses.append(last[0])
        groups.append(tr.last_step_groups)
        dev_ms.append(tr.last_step_ms)
        segs.append(tr.last_step_timings)
        real_tokens += int(lens_host[i % n_batches][0].sum())
        padded_tokens += B * lens_host[i % n_batches][1]
    barrier()
    dt_local = time.perf_counter() - t0
    e1 = meter.read_j()
    dt = rv.max_over_ranks(dt_local)
    launches = tr.launch_count - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(tr, args.dump_outputs, last, full)
    # ---- timed region 2: end to end through the host API (pinned host batches in, loss out) ----
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        losses.append(run(i, False)[0])
    barrier()
    dt_e2e = rv.max_over_ranks(time.perf_counter() - t0)
    clocks = sampler.stop()
    ev_ms = rv.max_over_ranks(float(np.mean(dev_ms)))
    mine = {"rank": rank, "device_ms_min": float(np.min(dev_ms)), "device_ms_median": float(np.median(dev_ms)),
            "device_ms_max": float(np.max(dev_ms)), "wall_ms_per_step": 1000.0 * dt_local / args.steps,
            "fwd_bwd_ms": float(np.median([s["fwd_bwd"] for s in segs])), "allreduce_ms": float(np.median([s["allreduce"] for s in segs])),
            "optimizer_ms": float(np.median([s["optimizer"] for s in segs])), "sm_mhz": clocks["sm_mhz"], "power_w": clocks.get("power_w"),
            "reasons": clocks["reasons"], "joules_per_step": ((e1 - e0) / args.steps) if (e0 is not None and e1 is not None) else None}
    ranks = rv.gather_objects(mine)
    real_all = rv.sum_over_ranks(float(real_tokens))
    padded_all = rv.sum_over_ranks(float(padded_tokens))

    tokens_per_step = B * S * world
    if varlen:  # the metric counts REAL tokens; the padded count is reported next to it
        value, e2e = real_all / dt, real_all / dt_e2e
    else:
        value, e2e = tokens_per_step * args.steps / dt, tokens_per_step * args.steps / dt_e2e
    if rank != 0:
        tr.close()
        return
    peaks = measured_peaks()
    gemms = time_step_gemms(torch, L) if args.config == "7b" else None
    tr.close()
    per_gpu_tflops = (value / world) * FLOP_PER_TOKEN / 1e12
    metric = {"13b_full": "tokens/sec Llama-2-13B full-parameter SFT seq2048", "small_full": "tokens/sec 0.6B Llama-arch full-parameter SFT seq2048",
              "7b": "tokens/sec Llama-2-7B LoRA SFT seq2048", "7b_varlen": "real (unpadded) tokens/sec Llama-2-7B LoRA SFT, variable-length rows <= 2048",
              "mistral7b_qlora": "tokens/sec Mistral-7B QLoRA nf4 r=32 seq4096", "tiny": "tokens/sec tiny-Llama smoke"}[args.config]
    workload = {"13b_full": "Llama-2-13B shape (L=40, d=5120, H=40, F=13824), FULL-parameter SFT: bf16 weights and gradients, per-layer NCCL reduce-scatter "
                            "overlapped with the backward pass, fp32 master weights + AdamW state sharded over the ranks, all-gather of the updated "
                            "weights; seq 2048, batch 4/GPU (BASELINE.json configs[3]; beyond the reference, NOT the headline metric)",
                "small_full": "Llama-architecture 0.6B (L=8, d=2048, F=5504), full-parameter SFT, seq 2048, batch 8/GPU (NOT the headline metric)",
                "7b": "Llama-2-7B (random-init N(0,0.02)) LoRA r=16 alpha=32 q_proj,v_proj, seq 2048, batch 8/GPU, "
                      "AdamW + clip 1.0 + linear schedule, bf16 compute / fp32 accumulate / fp32 adapters",
                "7b_varlen": "Llama-2-7B LoRA r=16 as in the headline config, but log-normal row lengths (median 512, clipped to [16, 2048]), "
                             "each batch padded to its longest row (128-rounded) with true row lengths passed to the step; NOT the headline metric",
                "mistral7b_qlora": "Mistral-7B shape (GQA 32/8, ffn 14336) QLoRA with packed NF4 base weights, r=32, seq 4096, batch 4/GPU "
                                   "(BASELINE.json configs[2]; NOT the headline metric, FLOP/token differs)",
                "tiny": "tiny-Llama smoke config (NOT the benchmark workload)"}[args.config]
    line = {
        "metric": metric, "value": value, "unit": "tokens/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": workload, "global_batch": B * world, "seq_len": S, "parallelism": f"dp{world}",
                   "l2": "per-step working set (13.5 GB weights + ~55 GB saved activations) >> 126 MB L2; no flush needed",
                   "recompute": "none (activations kept; the reference's gradient checkpointing is a memory knob, not math)",
                   "base_weight_bytes": base_bytes},
        "e2e": {"value": e2e, "unit": "tokens/s", "h2d_bytes_per_step": int(2 * padded_tokens / args.steps * 4 + (B * 4 if varlen else 0)),
                "d2h_bytes_per_step": 8, "ms_per_step": 1000.0 * dt_e2e / args.steps},
        "gpu_launches": int(launches),
        "device_ms_per_step": ev_ms,
        "clocks": {k: clocks[k] for k in ("sm_mhz", "sm_max_mhz", "reasons", "samples")},
        "ranks": ranks,
        "step_roofline": ({"bound": "tensor", "achieved": per_gpu_tflops, "peak": peaks["sustained"], "unit": "TFLOP/s",
                           "frac": per_gpu_tflops / peaks["sustained"], "flop_per_token": FLOP_PER_TOKEN,
                           "peak_src": peaks["src"] + " bf16_tflops_sustained"} if args.config == "7b" else None),
        "loss_first_last": [losses[0], losses[-1]] if losses else None,
    }
    if varlen:
        line["padded_tokens_per_s"] = padded_all / dt
        line["real_over_padded"] = real_all / padded_all
        # rows sorted by length and cut into groups by the library's cost model; each group runs at its own padded length
        line["length_groups_per_step"] = float(np.mean(groups))
        line["packed_steps"] = int(sum(1 for g in groups if g == 0))  # steps run packed: sequences back to back, one pass
        line["losses_first_batches"] = losses[:n_batches]
    if gemms:
        g = gemms["nn_dh2"]
        line["roofline"] = {"bound": "tensor", "achieved": g["tflops"], "peak": peaks["burst"], "unit": "TFLOP/s",
                            "frac": g["tflops"] / peaks["burst"], "traffic": GEMM_DRAM_BYTES.get("nn_dh2"),
                            "alg_bytes": g["alg_bytes"], "kernel": g["kernel"] + " (CTA-pair 256x256x64, cta_group::2; 31.8 % of the step)",
                            "shape_mnk": g["shape_mnk"], "ms": g["ms"], "peak_src": peaks["src"] + " bf16_tflops (burst)"}
        line["roofline_kernels"] = {k: {"kernel": v["kernel"], "shape_mnk": v["shape_mnk"], "ms": v["ms"], "tflops": v["tflops"],
                                        "frac": v["tflops"] / peaks["burst"], "alg_bytes": v["alg_bytes"], "traffic": GEMM_DRAM_BYTES.get(k)}
                                    for k, v in gemms.items()}
        # the same kernel under the 1 kW cap (0.2 s of back-to-back launches after 0.2 s of warm-up) against cuBLAS's sustained figure
        line["roofline"]["sustained"] = {"achieved": g["tflops_sustained"], "peak": peaks["sustained"], "frac": g["tflops_sustained"] / peaks["sustained"],
                                         "ms": g["ms_sustained"]}
    if args.cpu_baseline and args.config == "7b" and world == 1:
        line["cpu_baseline"] = cpu_arm(warmup=1, steps=1)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--config", default="7b", choices=["7b", "7b_varlen", "mistral7b_qlora", "13b_full", "small_full", "tiny"])
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last device-resident step "
                    "returned and the trainable parameters it left (rank 0) as DIR/<name>.npy, float32, <= 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs needs --impl native")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.warmup < 3 and args.impl == "native":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        print(json.dumps({"error": f"--gpus {args.gpus} needs torchrun (WORLD_SIZE={world})"}))
        sys.exit(2)
    run_native(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
