"""LoRA adapters on the MLP projections (gate_proj, up_proj, down_proj), alone or next to q/k/v_proj.

CPU: target bits and names, the reference forward against installed HF Llama with merged weights, the dropout-mask rule and
the PEFT files.  GPU (-m gpu): the K-extended fused-epilogue GEMMs and the dropout / SwiGLU-backward kernel per op, the training
step against the fp32 reference for every execution path, one Llama-2-7B-shaped layer and the worker end to end."""
import ctypes as C
import json
import math
import os

import numpy as np
import pytest
import torch

from oracle import llama_lora as O
from tests import lora_mlp_oracle as R
from tests.conftest import has_gpu

ALL6 = ("q_proj", "k_proj", "v_proj", "gate_proj", "up_proj", "down_proj")
MLP3 = ("gate_proj", "up_proj", "down_proj")


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def test_target_bits_accept_mlp_modules_and_refuse_o_proj():
    from datatunerx_b200 import lib as L
    tc = L.TrainConfig(micro_batch=1, seq_len=128, total_steps=1, lora_target=ALL6).to_c()
    assert tc.target_mask == 1 | 2 | 4 | 16 | 32 | 64
    assert L.TrainConfig(micro_batch=1, seq_len=128, total_steps=1, lora_target=MLP3).to_c().target_mask == 16 | 32 | 64
    with pytest.raises(L.DtxError) as e:
        L.TrainConfig(micro_batch=1, seq_len=128, total_steps=1, lora_target=("q_proj", "o_proj")).to_c()
    assert e.value.code == -5 and "o_proj" in str(e.value)


def _raw_create(lib, mask):
    from datatunerx_b200 import lib as L
    mc = L.ModelConfig(vocab=256, hidden=256, n_layers=1, n_heads=2, ffn=256).to_c()
    tc = L.TrainConfig(micro_batch=1, seq_len=128, total_steps=1, lora_dropout=0.0).to_c()
    tc.target_mask = mask
    h = C.c_void_p()
    rc = lib.dtx_trainer_create(C.byref(mc), C.byref(tc), 0, 0, 1, None, C.byref(h))
    if h:
        lib.dtx_trainer_destroy(h)
    return rc, (lib.dtx_last_global_error() or b"").decode()


def test_raw_create_refuses_o_proj_and_validates_mlp_bits(lib):
    rc, msg = _raw_create(lib, 1 | 8)
    assert rc == -5 and "o_proj" in msg, (rc, msg)  # DTX_ERR_UNSUPPORTED names the one module not implemented
    if torch.cuda.is_available():
        pytest.skip("GPU present: the MLP bits would create a trainer")
    for mask in (16 | 32 | 64, 1 | 2 | 4 | 16 | 32 | 64, 64):
        rc, msg = _raw_create(lib, mask)
        assert rc == -2, (mask, rc, msg)  # past validation: fails at the device (there is no CPU fallback)


def _merged_hf_logits(cfg, w, lora):
    """installed HF LlamaForCausalLM with W + (alpha/r) B A folded into every adapted module."""
    from transformers import LlamaConfig, LlamaForCausalLM
    merged = dict(w)
    s = cfg.lora_alpha / cfg.lora_r
    for k in lora:
        if k.endswith("lora_A.weight"):
            m = k[: -len(".lora_A.weight")]
            merged[m + ".weight"] = w[m + ".weight"] + s * lora[m + ".lora_B.weight"] @ lora[k]
    hc = LlamaConfig(vocab_size=cfg.vocab, hidden_size=cfg.hidden, intermediate_size=cfg.ffn, num_hidden_layers=cfg.n_layers,
                     num_attention_heads=cfg.n_heads, num_key_value_heads=cfg.n_kv_heads or cfg.n_heads, max_position_embeddings=4096,
                     rms_norm_eps=cfg.rms_eps, rope_theta=cfg.rope_theta, tie_word_embeddings=False, attn_implementation="eager")
    m = LlamaForCausalLM(hc).float()
    missing, unexpected = m.load_state_dict(merged, strict=False)
    assert not [k for k in missing if "rotary" not in k] and not unexpected
    return m.eval()


@pytest.mark.parametrize("targets", [MLP3, ("q_proj", "v_proj", "gate_proj", "up_proj", "down_proj"), ("down_proj",)])
def test_reference_matches_hf_llama_with_merged_adapters(targets):
    cfg = O.OracleConfig(vocab=512, hidden=256, n_layers=2, n_heads=2, ffn=384, lora_r=8, lora_alpha=16.0, lora_target=targets)
    w = O.init_base_weights(cfg, seed=7)
    lora = R.init_lora(cfg, seed=8)
    g = torch.Generator().manual_seed(9)
    for k in lora:  # non-zero B: the adapters change the output
        if "lora_B" in k:
            lora[k] = torch.randn(lora[k].shape, generator=g) * 0.02
    ids, _ = O.synthetic_batch(step=0, rank=0, batch=2, seq_len=64, vocab=cfg.vocab)
    t_ids = torch.from_numpy(ids).long()
    with torch.no_grad():
        ref = _merged_hf_logits(cfg, w, lora)(input_ids=t_ids).logits.float()
        got = R.forward_logits(cfg, w, lora, t_ids)
        base = O.forward_logits(cfg, w, {}, t_ids)
    assert torch.allclose(got, ref, atol=2e-5, rtol=1e-4)
    assert not torch.allclose(got, base, atol=1e-3)  # the adapters are live


def test_reference_shapes_and_fan_in():
    cfg = O.OracleConfig(vocab=512, hidden=256, n_layers=1, n_heads=2, ffn=384, lora_r=8, lora_target=ALL6)
    lora = R.init_lora(cfg, seed=3)
    p = "model.layers.0."
    assert lora[p + "mlp.gate_proj.lora_A.weight"].shape == (8, 256) and lora[p + "mlp.gate_proj.lora_B.weight"].shape == (384, 8)
    assert lora[p + "mlp.up_proj.lora_A.weight"].shape == (8, 256) and lora[p + "mlp.up_proj.lora_B.weight"].shape == (384, 8)
    assert lora[p + "mlp.down_proj.lora_A.weight"].shape == (8, 384) and lora[p + "mlp.down_proj.lora_B.weight"].shape == (256, 8)
    assert float(lora[p + "mlp.down_proj.lora_A.weight"].abs().max()) <= 1 / math.sqrt(384)
    assert float(lora[p + "mlp.down_proj.lora_A.weight"].abs().max()) > 0.9 / math.sqrt(384)
    assert not any(float(v.abs().max()) for k, v in lora.items() if "lora_B" in k)


def test_reference_equals_attention_oracle_on_qkv_targets():
    """q/k/v-only configurations: the same init stream, logits, loss and gradients as oracle/llama_lora.py, bit for bit."""
    cfg = O.OracleConfig(vocab=512, hidden=256, n_layers=2, n_heads=2, ffn=384, lora_r=8, lora_dropout=0.1,
                         lora_target=("q_proj", "k_proj", "v_proj"))
    w = O.init_base_weights(cfg, seed=7)
    a, b = O.init_lora(cfg, 8), R.init_lora(cfg, 8)
    assert a.keys() == b.keys() and all(torch.equal(a[k], b[k]) for k in a)
    ids, labels = O.synthetic_batch(step=0, rank=0, batch=2, seq_len=64, vocab=cfg.vocab)
    la, ga = O.OracleTrainer(cfg, w, a).loss_and_grads(ids, labels)
    lb, gb = R.OracleTrainer(cfg, w, b).loss_and_grads(ids, labels)
    assert la == lb and all(torch.equal(ga[k], gb[k]) for k in ga)


def test_dropout_mask_rule_for_mlp_targets():
    """Mask of a target = its position among the enabled targets in HF order; width = the module's input (ffn for down)."""
    cfg = O.OracleConfig(vocab=512, hidden=256, n_layers=2, n_heads=2, ffn=384, lora_dropout=0.25,
                         lora_target=("down_proj", "v_proj", "q_proj", "gate_proj"))
    masks = R.dropout_masks(cfg, (5, 1), 1, 96)
    key = O.dropout_key(cfg.seed, 5, 1, 1)
    order = {"q_proj": 0, "v_proj": 1, "gate_proj": 2, "down_proj": 3}
    assert set(masks) == set(order)
    assert masks["down_proj"].shape == (96, 384) and masks["gate_proj"].shape == (96, 256)
    for t, i in order.items():
        assert torch.equal(masks[t], O.dropout_mask(key, i, 96, 384 if t == "down_proj" else 256, 0.25)), t
    keep = float(masks["down_proj"].mean())
    assert 0.7 < keep < 0.8
    assert not torch.equal(masks["gate_proj"], masks["q_proj"])  # one independent mask per module
    # attention targets keep their masks when MLP targets are added
    qv = O.OracleConfig(vocab=512, hidden=256, n_layers=2, n_heads=2, ffn=384, lora_dropout=0.25, lora_target=("q_proj", "v_proj"))
    m_qv = R.dropout_masks(qv, (5, 1), 1, 96)
    assert torch.equal(m_qv["q_proj"], masks["q_proj"]) and torch.equal(m_qv["v_proj"], masks["v_proj"])


def _names_and_shapes(mc, tc):
    from datatunerx_b200 import lib as L
    tr = L.Trainer.__new__(L.Trainer)  # naming / shape arithmetic only: no device handle
    tr._h = C.c_void_p()
    tr.model, tr.train = mc, tc
    return {n: tr.adapter_shape(n) for n in tr.adapter_names()}


def test_peft_adapter_files_name_and_shape_mlp_adapters_as_peft(tmp_path):
    from transformers import LlamaConfig, LlamaForCausalLM
    from datatunerx_b200 import lib as L
    from datatunerx_b200.tuning import model_io
    targets = ["q_proj", "v_proj", "gate_proj", "up_proj", "down_proj"]
    mc = L.ModelConfig(vocab=400, hidden=256, n_layers=2, n_heads=2, n_kv_heads=1, ffn=768)
    tc = L.TrainConfig(micro_batch=1, seq_len=128, total_steps=1, lora_r=16, lora_target=tuple(targets))
    shapes = _names_and_shapes(mc, tc)
    # peft's LoraModel names every wrapped nn.Linear "base_model.model.<module path>" with lora_A [r, in], lora_B [out, r]
    hf = LlamaForCausalLM(LlamaConfig(vocab_size=400, hidden_size=256, intermediate_size=768, num_hidden_layers=2,
                                      num_attention_heads=2, num_key_value_heads=1))
    expect = {}
    for name, mod in hf.named_modules():
        if isinstance(mod, torch.nn.Linear) and name.rsplit(".", 1)[-1] in targets:
            expect[f"base_model.model.{name}.lora_A.weight"] = (16, mod.in_features)
            expect[f"base_model.model.{name}.lora_B.weight"] = (mod.out_features, 16)
    assert shapes == expect
    ad = {k: np.full(s, 0.5, np.float32) for k, s in shapes.items()}
    model_io.save_peft_adapter(str(tmp_path), ad, base_model="/models/tiny", r=16, alpha=32.0, dropout=0.1, target_modules=targets)
    cfg = json.load(open(tmp_path / "adapter_config.json"))
    assert cfg["target_modules"] == targets and cfg["r"] == 16
    back = {k: a for k, a, _ in model_io.iter_safetensors(str(tmp_path / "adapter_model.safetensors"))}
    assert {k: tuple(v.shape) for k, v in back.items()} == expect


def test_num_trainable_arithmetic_for_7b():
    """dtx_num_trainable's count: n_layers * sum r * (in + out) (the device trainer reports the same; checked on the GPU)."""
    from datatunerx_b200 import lib as L
    mc = L.ModelConfig.llama2_7b()
    for targets, n in ((ALL6, 35_782_656), (MLP3, 23_199_744), (("q_proj", "v_proj"), 8_388_608)):
        tc = L.TrainConfig(micro_batch=1, seq_len=128, total_steps=1, lora_r=16, lora_target=targets)
        assert sum(int(np.prod(s)) for s in _names_and_shapes(mc, tc).values()) == n, targets


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
def _gpu():
    if not has_gpu():
        pytest.skip("no GPU")
    from tests import gpu_checks as G
    return G


def _make_pair(steps=10, S=256, B=2, L_layers=2, heads=2, kv_heads=None, dropout=0.0, targets=ALL6, grad_accum=1, quant=False):
    from datatunerx_b200 import lib as L
    ocfg = O.OracleConfig(vocab=2048, hidden=128 * heads, n_layers=L_layers, n_heads=heads, n_kv_heads=kv_heads, ffn=768, lora_r=16,
                          lora_alpha=32.0, lr=1e-3, total_steps=steps, lora_dropout=dropout, lora_target=tuple(targets), grad_accum=grad_accum)
    mc = L.ModelConfig(vocab=2048, hidden=128 * heads, n_layers=L_layers, n_heads=heads, n_kv_heads=kv_heads, ffn=768)
    tc = L.TrainConfig(micro_batch=B, seq_len=S, total_steps=steps, lora_r=16, lora_alpha=32.0, lora_dropout=dropout, lr=1e-3,
                       lora_target=tuple(targets), grad_accum=grad_accum)
    w, lora = O.init_base_weights(ocfg, 1234), R.init_lora(ocfg, 4321)
    tr = L.Trainer(mc, tc)
    tr.load_state_dict({k: v.numpy() for k, v in w.items()})
    if quant:
        tr.quantize_base("int4")
        w = O.quantize_base_nf4(w)
    tr.load_state_dict({k: v.numpy() for k, v in lora.items()})
    return ocfg, R.OracleTrainer(ocfg, w, lora), tr


def _trainer_parity(steps=10, **kw):
    """10 optimizer steps against the fp32 reference: forward loss, step losses, grad-norms, adapters at the end."""
    ocfg, orc, tr = _make_pair(steps=steps, **kw)
    S, B, acc = tr.train.seq_len, tr.train.micro_batch, tr.train.grad_accum
    names = list(tr.adapter_names())
    assert len(names) == 2 * ocfg.n_layers * len(ocfg.lora_target)
    ids, labels = O.synthetic_batch(0, 0, B, S, ocfg.vocab)
    ref_eval = orc.eval_loss(ids, labels)
    e_eval = abs(tr.eval_loss(ids, labels) - ref_eval) / ref_eval
    assert e_eval < 1e-3, e_eval
    worst_l = worst_g = 0.0
    for s in range(steps):
        batches = [O.synthetic_batch(acc * s + i, 0, B, S, ocfg.vocab) for i in range(acc)]
        ref = orc.step(batches)
        losses = []
        for i, b in enumerate(batches):
            loss, gn, lr, stepped = tr.step(*b)
            assert stepped == (i == acc - 1)
            losses.append(loss)
        worst_l = max(worst_l, abs(float(np.mean(losses)) - ref.loss) / ref.loss)
        worst_g = max(worst_g, abs(gn - ref.grad_norm) / ref.grad_norm)
    ad, ref_ad = tr.export_adapter(), orc.state_dict()
    assert set(k.replace("base_model.model.", "") for k in ad) == set(ref_ad)
    worst_a = max(float(np.linalg.norm(v - ref_ad[k.replace("base_model.model.", "")]) /
                        max(np.linalg.norm(ref_ad[k.replace("base_model.model.", "")]), 1e-12)) for k, v in ad.items())
    moved = min(float(np.abs(v).max()) for k, v in ad.items() if "lora_B" in k)
    tr.close()
    res = {"eval": e_eval, "loss": worst_l, "gnorm": worst_g, "adapter": worst_a}
    assert worst_l < 1e-3 and worst_g < 3e-2 and worst_a < 0.15 and moved > 0, res
    return res


@pytest.mark.gpu
def test_gemm_kext_fused_epilogues_7b_widths():
    """The CTA-pair GEMM with a K-extension (the LoRA up-projection / input gradient) under the SwiGLU-forward, SwiGLU-backward
    (MN-major B2) and residual-add epilogues at Llama-2-7B widths (d = 4096, F = 11008, RP = 64)."""
    G = _gpu()
    from datatunerx_b200 import lib as L
    lib = L.load()
    M, d, F, RP = 1500, 4096, 11008, 64
    dev = G.DEV
    h2, wgu = G._rand(M, d, scale=0.5, seed=1), G._rand(2 * F, d, scale=0.02, seed=2)
    t_gu, b_gu = G._rand(M, RP, scale=0.5, seed=3), G._rand(2 * F, RP, scale=0.05, seed=4)
    gu = torch.empty(M, 2 * F, dtype=torch.bfloat16, device=dev)
    act = torch.empty(M, F, dtype=torch.bfloat16, device=dev)
    G.ok(lib.dtx_gemm_fused(G.P(h2), d, G.P(wgu), d, 0, G.P(t_gu), RP, G.P(b_gu), RP, RP, G.P(gu), 2 * F, G.P(act), F, None, 0, 0,
                            M, 2 * F, d, L.EPI_SWIGLU_FWD, G.STREAM()))
    ref_gu = h2.float() @ wgu.float().t() + t_gu.float() @ b_gu.float().t()
    gate, up = G._deinterleave_cols(ref_gu, F)
    torch.cuda.synchronize()
    e_fwd = (G.rel_err(gu, ref_gu), G.rel_err(act, torch.nn.functional.silu(gate) * up))
    # backward: d(gate|up) from d(act) = dx * Wdown + dt * A_dn (A_dn [RP, F]: MN-major B2)
    dx, wdown = G._rand(M, d, scale=0.5, seed=5), G._rand(d, F, scale=0.02, seed=6)
    dt, a_dn = G._rand(M, RP, scale=0.5, seed=7), G._rand(RP, F, scale=0.05, seed=8)
    dgu = torch.empty(M, 2 * F, dtype=torch.bfloat16, device=dev)
    G.ok(lib.dtx_gemm_fused(G.P(dx), d, G.P(wdown), F, 1, G.P(dt), RP, G.P(a_dn), F, RP, G.P(dgu), 2 * F, G.P(gu), 2 * F, None, 0, 0,
                            M, F, d, L.EPI_SWIGLU_BWD, G.STREAM()))
    dact = dx.float() @ wdown.float() + dt.float() @ a_dn.float()
    g_f, u_f = G._deinterleave_cols(gu.float(), F)
    sg = torch.sigmoid(g_f)
    ref_dg, ref_du = dact * u_f * (sg + g_f * sg * (1 - sg)), dact * g_f * sg
    got_dg, got_du = G._deinterleave_cols(dgu.float(), F)
    torch.cuda.synchronize()
    e_bwd = (G.rel_err(got_dg, ref_dg), G.rel_err(got_du, ref_du))
    # down projection with the residual: x_next = x_mid + act * Wdown^T + t_dn * B_dn^T  (K = F)
    t_dn, b_dn, x_mid = G._rand(M, RP, scale=0.5, seed=9), G._rand(d, RP, scale=0.05, seed=10), G._rand(M, d, scale=1.0, seed=11)
    xn = torch.empty(M, d, dtype=torch.bfloat16, device=dev)
    G.ok(lib.dtx_gemm_bf16(G.P(act), F, 0, G.P(wdown), F, 0, G.P(t_dn), RP, G.P(b_dn), RP, RP, G.P(xn), d, G.P(x_mid), d,
                           M, d, F, L.EPI_BF16_ADD, 1, 0, G.STREAM()))
    ref_xn = x_mid.float() + act.float() @ wdown.float().t() + t_dn.float() @ b_dn.float().t()
    torch.cuda.synchronize()
    e_add = G.rel_err(xn, ref_xn)
    assert max(e_fwd) < 1e-2 and max(e_bwd) < 2e-2 and e_add < 1e-2, (e_fwd, e_bwd, e_add)


@pytest.mark.gpu
@pytest.mark.parametrize("interleaved", [0, 1])
def test_swiglu_bwd_lora_dropout_kernel(interleaved):
    """dgu = SwiGLU backward of dact + mask o g / (1 - p), the mask regenerated exactly as dtx_lora_dropout_fwd draws it."""
    G = _gpu()
    from datatunerx_b200 import lib as L
    lib = L.load()
    M, F, p, key = 300, 768, 0.1, 0x1234_5678_9ABC_DEF1
    dact, g, gu = G._rand(M, F, seed=1), G._rand(M, F, seed=2), G._rand(M, 2 * F, seed=3)
    ones = torch.ones(M, F, dtype=torch.bfloat16, device="cuda")
    mask = torch.empty_like(ones)
    G.ok(lib.dtx_lora_dropout_fwd(G.P(ones), G.P(mask), M, F, 1, p, key, G.STREAM()))  # kept: 1/(1-p), dropped: 0
    dgu = torch.empty(M, 2 * F, dtype=torch.bfloat16, device="cuda")
    G.ok(lib.dtx_swiglu_bwd_lora_dropout(G.P(dact), G.P(g), G.P(gu), G.P(dgu), M, F, interleaved, p, key, G.STREAM()))
    torch.cuda.synchronize()
    keep = (mask.float() > 0).float()
    d_act = dact.float() + keep * g.float() / (1 - p)
    if interleaved:
        gate, up = G._deinterleave_cols(gu.float(), F)
        got_g, got_u = G._deinterleave_cols(dgu.float(), F)
    else:
        gate, up = gu.float()[:, :F], gu.float()[:, F:]
        got_g, got_u = dgu.float()[:, :F], dgu.float()[:, F:]
    s = torch.sigmoid(gate)
    assert G.rel_err(got_g, d_act * up * (s + gate * s * (1 - s))) < 1e-2
    assert G.rel_err(got_u, d_act * gate * s) < 1e-2
    assert 0.85 < float(keep.mean()) < 0.95


TINY_CASES = {
    "mlp_only": dict(targets=MLP3),
    "qv_mlp": dict(targets=("q_proj", "v_proj") + MLP3),
    "all6_gqa": dict(heads=4, kv_heads=2),
    "all6_dropout": dict(dropout=0.1),
    "all6_unfused": dict(),
    "all6_single_cta": dict(),
    "all6_grad_accum": dict(grad_accum=2, steps=5),
    "all6_qlora": dict(quant=True),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(TINY_CASES))
def test_trainer_tiny_mlp_targets(case):
    _gpu()
    from datatunerx_b200 import lib as L
    opts = {"all6_unfused": {"fused_epilogues": 0}, "all6_single_cta": {"gemm_pair_kernel": 0, "fused_epilogues": 0}}.get(case, {})
    for k, v in opts.items():
        L.set_option(k, v)
    try:
        _trainer_parity(**TINY_CASES[case])
    finally:
        for k in opts:
            L.set_option(k, 1)


@pytest.mark.gpu
def test_num_trainable_on_device():
    _gpu()
    from datatunerx_b200 import lib as L
    ocfg, _, tr = _make_pair(targets=ALL6, L_layers=1)
    n = tr.num_trainable
    tr.close()
    assert n == sum(int(np.prod(s)) for s in _names_and_shapes(tr.model, tr.train).values())


@pytest.mark.gpu
def test_layer_7b_shape_all_targets(B=2, S=2048):
    """One Llama-2-7B-shaped layer with all six adapters (B randomised) against the fp32 reference: eval loss, step loss,
    grad-norm and every adapter gradient; then a ragged batch (2048 + 700 tokens) as two length groups and packed."""
    _gpu()
    from datatunerx_b200 import lib as L
    ocfg = O.OracleConfig(vocab=32000, hidden=4096, n_layers=1, n_heads=32, ffn=11008, lora_r=16, lora_alpha=32.0, lr=1e-4, total_steps=100,
                          lora_target=ALL6)
    mc = L.ModelConfig(vocab=32000, hidden=4096, n_layers=1, n_heads=32, ffn=11008)
    tc = L.TrainConfig(micro_batch=B, seq_len=S, total_steps=100, lora_r=16, lora_alpha=32.0, lora_dropout=0.0, lr=1e-4, lora_target=ALL6)
    w, lora = O.init_base_weights(ocfg, 1234), R.init_lora(ocfg, 4321)
    g = torch.Generator().manual_seed(99)
    for k in lora:
        if "lora_B" in k:
            lora[k] = torch.randn(lora[k].shape, generator=g) * 0.01
    tr = L.Trainer(mc, tc)
    tr.load_state_dict({k: v.numpy() for k, v in w.items()})
    tr.load_state_dict({k: v.numpy() for k, v in lora.items()})
    orc = R.OracleTrainer(ocfg, w, lora)

    def rel_errs(got, ref):
        return {k.split("layers.0.")[1]: float(np.linalg.norm(v - ref[k.replace("base_model.model.", "")].numpy()) /
                                               max(np.linalg.norm(ref[k.replace("base_model.model.", "")].numpy()), 1e-12)) for k, v in got.items()}

    ids, labels = O.synthetic_batch(0, 0, B, S, ocfg.vocab)
    ref_loss, g_ref = orc.loss_and_grads(ids, labels)
    e_eval = abs(tr.eval_loss(ids, labels) - ref_loss) / ref_loss
    loss, gn, _, _ = tr.step(ids, labels)
    ref_norm = math.sqrt(sum(float((v.double() ** 2).sum()) for v in g_ref.values()))
    errs = rel_errs(tr.export_adapter(grads=True), g_ref)
    res = {"eval": e_eval, "loss": abs(loss - ref_loss) / ref_loss, "gnorm": abs(gn - ref_norm) / ref_norm, "grads": errs}
    assert len(errs) == 12 and res["eval"] < 1e-3 and res["loss"] < 1e-3 and res["gnorm"] < 3e-2 and max(errs.values()) < 4e-2, res
    lens = np.array([S, 700], dtype=np.int32)
    ids2, labels2 = O.synthetic_batch(1, 0, B, S, ocfg.vocab)
    ids2[1, 700:] = 0
    labels2[1, 700:] = -100
    ref2, g2 = orc.loss_and_grads(ids2, labels2)
    for mode in ("groups", "packed"):
        tr.load_state_dict({k: v.numpy() for k, v in lora.items()})
        if mode == "groups":
            L.set_option("varlen_split", 2)
        try:
            loss2, _, _, _ = tr.step(ids2, labels2, lens)
            groups = tr.last_step_groups
        finally:
            L.set_option("varlen_split", 1)
        e2 = rel_errs(tr.export_adapter(grads=True), g2)
        res[mode] = {"groups": groups, "loss": abs(loss2 - ref2) / ref2, "grads": max(e2.values())}
        assert groups == (2 if mode == "groups" else 0) and res[mode]["loss"] < 1e-3 and res[mode]["grads"] < 4e-2, res
    tr.close()


@pytest.mark.gpu
def test_worker_end_to_end_with_mlp_targets():
    """The worker behind the controller's command line with --lora_target q_proj,v_proj,gate_proj,up_proj,down_proj."""
    G = _gpu()
    import importlib
    import shlex
    import shutil
    import tempfile
    from datatunerx_b200.tuning import model_io, parser as TP
    targets = ["q_proj", "v_proj", "gate_proj", "up_proj", "down_proj"]
    tmp = tempfile.mkdtemp(prefix="dtx_e2e_mlp_")
    try:
        mdir, store = os.path.join(tmp, "model"), os.path.join(tmp, "storage")
        os.makedirs(mdir)
        gold = os.path.join(os.path.dirname(__file__), "golden")
        shutil.copy(os.path.join(gold, "tiny_tokenizer.json"), os.path.join(mdir, "tokenizer.json"))
        json.dump({"tokenizer_class": "PreTrainedTokenizerFast", "bos_token": "<s>", "eos_token": "</s>", "unk_token": "<unk>"},
                  open(os.path.join(mdir, "tokenizer_config.json"), "w"))
        ocfg = O.OracleConfig(vocab=400, hidden=256, n_layers=2, n_heads=2, ffn=768)
        json.dump({"architectures": ["LlamaForCausalLM"], "vocab_size": 400, "hidden_size": 256, "intermediate_size": 768,
                   "num_hidden_layers": 2, "num_attention_heads": 2, "num_key_value_heads": 2, "rms_norm_eps": 1e-5, "rope_theta": 10000.0,
                   "max_position_embeddings": 4096, "model_type": "llama"}, open(os.path.join(mdir, "config.json"), "w"))
        model_io.write_safetensors(os.path.join(mdir, "model.safetensors"), {k: v.numpy() for k, v in O.init_base_weights(ocfg, 7).items()})
        csv_path = os.path.join(tmp, "train.csv")
        with open(csv_path, "w") as f:
            f.write("q,a\n")
            for i in range(48):
                f.write(f"What is {i} plus {i}?,The answer is {2 * i}.\n")
        ckpt_file = os.path.join(tmp, "checkpoint_path")
        os.environ["DTX_CHECKPOINT_PATH_FILE"] = ckpt_file
        from datatunerx_b200.tuning import train as TT
        importlib.reload(TT)
        entry = TP.controller_entrypoint(mdir, csv_path, validate_file=csv_path, columns='{"instruction":"q","response":"a"}',
                                         scheduler="linear", optimizer="adamw_hf", lora_r="16", lora_alpha="32", lora_dropout="0.0",
                                         learning_rate="1e-3", epochs=2, block_size=256, batch_size=4, grad_acc_steps=1,
                                         num_workers=1, storage_path=store, uid="e2e")
        assert "--lora_target q_proj,v_proj " in entry
        entry = entry.replace("--lora_target q_proj,v_proj ", "--lora_target " + ",".join(targets) + " ")
        cwd = os.getcwd()
        os.chdir(tmp)
        try:
            rc = TT.main(shlex.split(entry)[2:])
        finally:
            os.chdir(cwd)
        assert rc == 0, f"worker exit status {rc}"
        ckpt = open(ckpt_file).read()
        cfg = json.load(open(os.path.join(ckpt, "adapter_config.json")))
        assert cfg["target_modules"] == targets, cfg
        ad = {k: np.array(a) for k, a, _ in model_io.iter_safetensors(os.path.join(ckpt, "adapter_model.safetensors"))}
        assert len(ad) == 20 and all(np.isfinite(v).all() for v in ad.values())
        for k, v in ad.items():
            mod = k.split(".lora_")[0].rsplit(".", 1)[-1]
            d_in, d_out = R.linear_dims(ocfg, mod)
            assert k.startswith("base_model.model.model.layers.") and (".mlp." in k) == (mod in MLP3), k
            assert v.shape == ((16, d_in) if "lora_A" in k else (d_out, 16)), (k, v.shape)
        assert all(np.abs(v).max() > 0 for k, v in ad.items() if "lora_B" in k), "every B adapter must have moved"
        logs = [json.loads(l) for l in open(os.path.join(tmp, "result", "watch", "trainer_log.jsonl"))]
        assert logs[-1]["loss"] < logs[0]["loss"], logs
    finally:
        os.environ.pop("DTX_CHECKPOINT_PATH_FILE", None)
        shutil.rmtree(tmp, ignore_errors=True)
