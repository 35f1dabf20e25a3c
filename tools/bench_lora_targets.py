"""Step time of the LoRA trainer by adapter target set, on one GPU.

Configurations (Llama-2-7B, r = 16, batch 8 x 2048 tokens, random base weights, device-resident synthetic batches):
  q,v (the headline bench config) | q,k,v,gate,up,down (dropout 0) | the same with dropout 0.1 | gate,up,down
and the Mistral-7B QLoRA shape of bench.py (NF4 base, GQA 32/8, ffn 14336, batch 4 x 4096) with all six targets at r = 32.
Only one 7B trainer fits next to another's activations, so each round creates, warms up, times and frees every configuration
in turn; `--rounds` rounds alternate them.  Times come from the trainer's device events (dtx_last_step_ms).  One JSON line per
(configuration, round), then one summary line per configuration; the device name and power limit are read in the same run.

usage: python tools/bench_lora_targets.py [--steps 5] [--warmup 2] [--rounds 2] [--configs qv,all6,...] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ALL6 = ("q_proj", "k_proj", "v_proj", "gate_proj", "up_proj", "down_proj")
CONFIGS = {
    "qv": dict(targets=("q_proj", "v_proj"), dropout=0.0),
    "all6": dict(targets=ALL6, dropout=0.0),
    "all6_dropout": dict(targets=ALL6, dropout=0.1),
    "mlp3": dict(targets=("gate_proj", "up_proj", "down_proj"), dropout=0.0),
    "mistral7b_qlora_all6": dict(targets=ALL6, dropout=0.0, mistral=True),
}


def gpu_identity():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True, check=False).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def run_config(name, steps, warmup):
    import numpy as np
    import torch
    from datatunerx_b200 import lib as L
    from datatunerx_b200.tuning.synthetic import synthetic_batch
    c = CONFIGS[name]
    if c.get("mistral"):
        mc = L.ModelConfig(vocab=32000, hidden=4096, n_layers=32, n_heads=32, n_kv_heads=8, ffn=14336, max_seq=32768, sliding_window=4096)
        B, S, r, quant = 4, 4096, 32, "int4"
    else:
        mc, B, S, r, quant = L.ModelConfig.llama2_7b(), 8, 2048, 16, None
    tc = L.TrainConfig(micro_batch=B, seq_len=S, total_steps=100, lora_r=r, lora_alpha=32.0, lora_dropout=c["dropout"], lr=1e-4,
                       lora_target=c["targets"])
    tr = L.Trainer(mc, tc)
    try:
        tr.init_random_weights(1234)
        if quant:
            tr.quantize_base(quant)
        tr.init_lora(4321)
        dev = []
        for i in range(2):
            ids, lab = synthetic_batch(i, 0, B, S, mc.vocab)
            dev.append((torch.from_numpy(ids).cuda(), torch.from_numpy(lab).cuda()))
        torch.cuda.synchronize()
        for i in range(warmup):
            tr.step_ptr(dev[i % 2][0].data_ptr(), dev[i % 2][1].data_ptr(), on_device=True)
        l0 = tr.launch_count
        ms, losses = [], []
        for i in range(steps):
            loss, _, _, _ = tr.step_ptr(dev[i % 2][0].data_ptr(), dev[i % 2][1].data_ptr(), on_device=True)
            ms.append(tr.last_step_ms)
            losses.append(loss)
        launches = (tr.launch_count - l0) / steps
        assert all(np.isfinite(losses)), losses
        med = float(np.median(ms))
        return {"config": name, "targets": ",".join(t.replace("_proj", "") for t in c["targets"]), "lora_r": r,
                "lora_dropout": c["dropout"], "batch": B, "seq_len": S, "ms_per_step_median": round(med, 3),
                "ms_per_step_all": [round(x, 3) for x in ms], "tokens_per_s": round(B * S / (med / 1000.0), 1),
                "trainable_params": tr.num_trainable, "launches_per_step": launches, "loss_last": losses[-1]}
    finally:
        tr.close()
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--configs", default=",".join(CONFIGS))
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: this benchmark only measures on the GPU"}))
        return 2
    names = args.configs.split(",")
    gpu = gpu_identity()
    lines, by = [], {n: [] for n in names}
    for rnd in range(args.rounds):
        for n in names:
            t0 = time.time()
            res = run_config(n, args.steps, args.warmup)
            res.update({"round": rnd, "gpu": gpu, "wall_s": round(time.time() - t0, 1)})
            by[n].append(res)
            lines.append(res)
            print(json.dumps(res), flush=True)
    base = min(r["ms_per_step_median"] for r in by.get("qv", [])) if by.get("qv") else None
    for n in names:
        best = min(r["ms_per_step_median"] for r in by[n])
        s = {"summary": n, "gpu": gpu, "ms_per_step_best_round": best, "ms_per_step_rounds": [r["ms_per_step_median"] for r in by[n]],
             "tokens_per_s": round(by[n][0]["batch"] * by[n][0]["seq_len"] / (best / 1000.0), 1),
             "trainable_params": by[n][0]["trainable_params"], "launches_per_step": by[n][0]["launches_per_step"]}
        if base and not CONFIGS[n].get("mistral"):
            s["vs_qv"] = round(best / base, 4)
        lines.append(s)
        print(json.dumps(s), flush=True)
    if args.out:
        with open(args.out, "a") as f:
            for l in lines:
                f.write(json.dumps(l) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
