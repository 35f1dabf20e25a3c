"""ctypes binding of libdtxtune.so — the C ABI declared in include/dtxtune.h.

This is the reference-side stub a maintainer would add (INTEGRATION.md shows the cgo twin).  It does
no arithmetic: every call lands in the sm_100a kernels.  There is no CPU fallback — if the shared
library is missing, or no CUDA device is visible, the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import Dict, Iterable, Optional, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# DTX_LIB_PATH selects another build of the same library (e.g. the clock64()-instrumented libdtxtune_timing.so of tools/attn_timing.py)
LIB_PATH = os.environ.get("DTX_LIB_PATH") or os.path.join(_HERE, "libdtxtune.so")

DTX_F32, DTX_BF16, DTX_F16 = 0, 1, 2
SCHED = {"linear": 0, "cosine": 1, "constant": 2, "constant_with_warmup": 3}
# LoRA target bits in HF module order (include/dtxtune.h); bit 8 (o_proj) is reserved: its adapter is not implemented
TARGET_BITS = {"q_proj": 1, "k_proj": 2, "v_proj": 4, "gate_proj": 16, "up_proj": 32, "down_proj": 64}
MLP_TARGETS = ("gate_proj", "up_proj", "down_proj")
EPI_BF16, EPI_F32, EPI_BF16_ADD, EPI_ROPE, EPI_SWIGLU_FWD, EPI_SWIGLU_BWD = 0, 1, 2, 3, 4, 5
STEP_FORCE = 1


class DtxError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libdtxtune error {code}: {msg}")
        self.code = code


class ModelCfg(C.Structure):
    _fields_ = [("vocab", C.c_int32), ("hidden", C.c_int32), ("n_layers", C.c_int32), ("n_heads", C.c_int32),
                ("n_kv_heads", C.c_int32), ("head_dim", C.c_int32), ("ffn", C.c_int32), ("rms_eps", C.c_float),
                ("rope_theta", C.c_float), ("max_seq", C.c_int32), ("sliding_window", C.c_int32)]


class TrainCfg(C.Structure):
    _fields_ = [("lora_r", C.c_int32), ("lora_alpha", C.c_float), ("lora_dropout", C.c_float),
                ("target_mask", C.c_uint32), ("lr", C.c_float), ("weight_decay", C.c_float), ("beta1", C.c_float),
                ("beta2", C.c_float), ("eps", C.c_float), ("max_grad_norm", C.c_float), ("sched", C.c_int32),
                ("warmup_steps", C.c_int32), ("total_steps", C.c_int32), ("grad_accum", C.c_int32),
                ("micro_batch", C.c_int32), ("seq_len", C.c_int32), ("seed", C.c_uint64), ("full_finetune", C.c_int32),
                ("reserved", C.c_int32)]


# every symbol include/dtxtune.h declares (tests/test_abi.py checks the .so exports all of them)
ABI_SYMBOLS = [
    "dtx_abi_version", "dtx_last_global_error", "dtx_last_error", "dtx_trainer_create", "dtx_trainer_destroy",
    "dtx_get_nccl_unique_id", "dtx_load_tensor", "dtx_init_random_weights", "dtx_init_lora", "dtx_quantize_base", "dtx_step",
    "dtx_step_device", "dtx_eval_loss", "dtx_allreduce_host", "dtx_export_adapter", "dtx_export_adapter_grad", "dtx_export_weight", "dtx_num_trainable", "dtx_launch_count",
    "dtx_base_weight_bytes", "dtx_last_step_ms", "dtx_last_step_timings", "dtx_last_step_groups", "dtx_plan_length_groups", "dtx_plan_packed_rows", "dtx_lr_lambda", "dtx_set_option", "dtx_gemm_bf16",
    "dtx_gemm_fused", "dtx_embedding_fwd", "dtx_rmsnorm_fwd", "dtx_rmsnorm_bwd",
    "dtx_rope_table", "dtx_rope_qk", "dtx_swiglu_fwd", "dtx_swiglu_bwd", "dtx_lora_dropout_fwd", "dtx_lora_dropout_bwd_add",
    "dtx_swiglu_bwd_lora_dropout", "dtx_nf4_roundtrip", "dtx_nf4_pack", "dtx_nf4_dequant", "dtx_cross_entropy", "dtx_sumsq", "dtx_adamw",
    "dtx_attn_fwd", "dtx_attn_bwd",
]

_lib: Optional[C.CDLL] = None


def load() -> C.CDLL:
    """dlopen libdtxtune.so (built in-tree by datatunerx_b200/csrc/Makefile).  Fails loudly."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DtxError(-2, f"{LIB_PATH} not found: build it with `make -C datatunerx_b200/csrc` "
                           "(python -c 'import __graft_entry__ as g; g.build()'); there is no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float
    lib.dtx_abi_version.restype = i32
    lib.dtx_last_global_error.restype = C.c_char_p
    lib.dtx_last_error.restype = C.c_char_p
    lib.dtx_last_error.argtypes = [vp]
    lib.dtx_trainer_create.argtypes = [C.POINTER(ModelCfg), C.POINTER(TrainCfg), i32, i32, i32, vp, C.POINTER(vp)]
    lib.dtx_trainer_destroy.argtypes = [vp]
    lib.dtx_trainer_destroy.restype = None
    lib.dtx_get_nccl_unique_id.argtypes = [vp]
    lib.dtx_load_tensor.argtypes = [vp, C.c_char_p, vp, i32, C.POINTER(i64), i32]
    lib.dtx_init_random_weights.argtypes = [vp, C.c_uint64]
    lib.dtx_init_lora.argtypes = [vp, C.c_uint64]
    lib.dtx_quantize_base.argtypes = [vp, i32]
    lib.dtx_nf4_roundtrip.argtypes = [vp, i64, vp]
    lib.dtx_nf4_pack.argtypes = [vp, vp, vp, i64, vp]
    lib.dtx_nf4_dequant.argtypes = [vp, vp, vp, i64, vp]
    lib.dtx_step.argtypes = [vp, vp, vp, vp, i32, i32, C.POINTER(f32), C.POINTER(f32), C.POINTER(f32), C.POINTER(i32)]
    lib.dtx_step_device.argtypes = [vp, vp, vp, vp, i32, i32, C.POINTER(f32), C.POINTER(f32), C.POINTER(f32), C.POINTER(i32)]
    lib.dtx_eval_loss.argtypes = [vp, vp, vp, vp, i32, C.POINTER(f32), vp, vp]
    lib.dtx_allreduce_host.argtypes = [vp, vp, i32]
    lib.dtx_base_weight_bytes.argtypes = [vp]
    lib.dtx_base_weight_bytes.restype = i64
    lib.dtx_last_step_timings.argtypes = [vp, vp]
    lib.dtx_last_step_groups.argtypes = [vp]
    lib.dtx_plan_length_groups.argtypes = [vp, i32, i32, vp, i32, vp, vp, vp]
    lib.dtx_plan_packed_rows.argtypes = [i32, vp, i32, vp]
    lib.dtx_gemm_fused.argtypes = [vp, i64, vp, i64, i32, vp, i64, vp, i64, i32, vp, i64, vp, i64, vp, i32, i32, i32, i32, i32,
                                   i32, vp]
    lib.dtx_export_adapter.argtypes = [vp, C.c_char_p, vp, i64]
    lib.dtx_export_adapter_grad.argtypes = [vp, C.c_char_p, vp, i64]
    lib.dtx_export_weight.argtypes = [vp, C.c_char_p, vp, i64, i32]
    lib.dtx_num_trainable.argtypes = [vp]
    lib.dtx_num_trainable.restype = i64
    lib.dtx_launch_count.argtypes = [vp]
    lib.dtx_launch_count.restype = i64
    lib.dtx_last_step_ms.argtypes = [vp]
    lib.dtx_last_step_ms.restype = f32
    lib.dtx_lr_lambda.argtypes = [i32, i32, i32, i32]
    lib.dtx_lr_lambda.restype = C.c_double
    lib.dtx_set_option.argtypes = [C.c_char_p, i32]
    lib.dtx_gemm_bf16.argtypes = [vp, i64, i32, vp, i64, i32, vp, i64, vp, i64, i32, vp, i64, vp, i64, i32, i32, i32, i32,
                                  i32, i32, vp]
    lib.dtx_embedding_fwd.argtypes = [vp, vp, vp, i32, i32, i32, vp]
    lib.dtx_rmsnorm_fwd.argtypes = [vp, vp, vp, vp, i32, i32, f32, vp]
    lib.dtx_rmsnorm_bwd.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, vp]
    lib.dtx_rope_table.argtypes = [vp, i32, i32, f32, vp]
    lib.dtx_rope_qk.argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, vp]
    lib.dtx_swiglu_fwd.argtypes = [vp, vp, i32, i32, vp]
    lib.dtx_swiglu_bwd.argtypes = [vp, vp, vp, i32, i32, vp]
    lib.dtx_lora_dropout_fwd.argtypes = [vp, vp, i32, i32, i32, f32, C.c_uint64, vp]
    lib.dtx_lora_dropout_bwd_add.argtypes = [vp, vp, i32, i32, i32, f32, C.c_uint64, vp]
    lib.dtx_swiglu_bwd_lora_dropout.argtypes = [vp, vp, vp, vp, i32, i32, i32, f32, C.c_uint64, vp]
    lib.dtx_cross_entropy.argtypes = [vp, i64, vp, vp, vp, vp, vp, i64, vp, i32, i32, i32, vp]
    lib.dtx_sumsq.argtypes = [vp, i64, vp, vp, vp]
    lib.dtx_adamw.argtypes = [vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, i32, f32, vp, f32, vp, vp]
    lib.dtx_attn_fwd.argtypes = [vp, vp, vp, i32, i32, i32, i32, f32, vp, i32, vp]
    lib.dtx_attn_bwd.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, f32, vp, i32, vp, i32, vp]
    for name in ABI_SYMBOLS:
        fn = getattr(lib, name)
        if fn.restype is C.c_int:  # default: all status-returning entry points
            fn.restype = i32
    _lib = lib
    return lib


def check(code: int, handle=None) -> None:
    if code != 0:
        lib = load()
        msg = lib.dtx_last_error(handle) if handle else lib.dtx_last_global_error()
        raise DtxError(code, (msg or b"").decode("utf-8", "replace"))


def set_option(name: str, value: int) -> None:
    check(load().dtx_set_option(name.encode(), value))


def plan_packed_rows(seq_lens, seq_len_batch: int):
    """The packed layout of a ragged micro-batch (host arithmetic inside the library): (first row of every sequence + total rows,
    whether packing saves rows over the padded rectangle)."""
    lens = np.ascontiguousarray(seq_lens, dtype=np.int32)
    starts = np.zeros(int(lens.shape[0]) + 1, np.int32)
    rc = load().dtx_plan_packed_rows(int(lens.shape[0]), lens.ctypes.data_as(C.c_void_p), seq_len_batch, starts.ctypes.data_as(C.c_void_p))
    if rc < 0:
        raise DtxError(rc, "dtx_plan_packed_rows")
    return starts.tolist(), bool(rc)


def plan_length_groups(model: "ModelConfig", seq_lens, seq_len_batch: int, n_sms: int = 0):
    """The partition dtx_step chooses for a ragged LoRA micro-batch (host arithmetic inside the library, no GPU needed):
    a list of (rows, padded_length) - rows are indices into the micro-batch, longest first."""
    lens = np.ascontiguousarray(seq_lens, dtype=np.int32)
    B = int(lens.shape[0])
    order, start, glen = np.zeros(B, np.int32), np.zeros(B + 1, np.int32), np.zeros(B, np.int32)
    mc = model.to_c()
    n = load().dtx_plan_length_groups(C.byref(mc), B, n_sms, lens.ctypes.data_as(C.c_void_p), seq_len_batch,
                                      order.ctypes.data_as(C.c_void_p), start.ctypes.data_as(C.c_void_p), glen.ctypes.data_as(C.c_void_p))
    if n < 1:
        raise DtxError(n, "dtx_plan_length_groups")
    return [([int(r) for r in order[start[g]:start[g + 1]]], int(glen[g])) for g in range(n)]


def lr_lambda(sched: str, step: int, warmup: int, total: int) -> float:
    """HF get_scheduler multiplier — host arithmetic inside the library, usable without a GPU."""
    return float(load().dtx_lr_lambda(SCHED[sched], step, warmup, total))


@dataclass
class ModelConfig:
    vocab: int
    hidden: int
    n_layers: int
    n_heads: int
    ffn: int
    n_kv_heads: Optional[int] = None
    head_dim: int = 128
    rms_eps: float = 1e-5
    rope_theta: float = 10000.0
    max_seq: int = 4096
    sliding_window: int = 0            # Mistral config.json `sliding_window`; 0 = none

    @staticmethod
    def llama2_7b() -> "ModelConfig":
        return ModelConfig(vocab=32000, hidden=4096, n_layers=32, n_heads=32, ffn=11008)

    def to_c(self) -> ModelCfg:
        return ModelCfg(self.vocab, self.hidden, self.n_layers, self.n_heads, self.n_kv_heads or self.n_heads,
                        self.head_dim, self.ffn, self.rms_eps, self.rope_theta, self.max_seq, int(self.sliding_window or 0))


@dataclass
class TrainConfig:
    micro_batch: int
    seq_len: int
    total_steps: int
    lora_r: int = 8                     # cmd/tuning/parser.py:138-141
    lora_alpha: float = 32.0            # parser.py:142-145
    lora_dropout: float = 0.1           # parser.py:146-149
    lora_target: Tuple[str, ...] = ("q_proj", "v_proj")  # finetune_controller.go:482
    lr: float = 5e-5                    # HF TrainingArguments default
    weight_decay: float = 0.0
    beta1: float = 0.9
    beta2: float = 0.999
    eps: float = 1e-8
    max_grad_norm: float = 1.0
    sched: str = "linear"
    warmup_steps: int = 0               # --warmup_ratio is dropped by the reference (train.py:204)
    grad_accum: int = 1
    seed: int = 42
    full_finetune: bool = False         # every weight trains, no adapters (BASELINE.json configs[3]; beyond the reference)

    def to_c(self) -> TrainCfg:
        mask = 0
        for t in self.lora_target:
            if t not in TARGET_BITS:
                raise DtxError(-5, f"lora_target {t!r} is not implemented natively (q_proj,k_proj,v_proj,gate_proj,up_proj,down_proj "
                                   "are; o_proj is the one linear module whose adapter is not)")
            mask |= TARGET_BITS[t]
        return TrainCfg(self.lora_r, self.lora_alpha, self.lora_dropout, mask, self.lr, self.weight_decay, self.beta1,
                        self.beta2, self.eps, self.max_grad_norm, SCHED[self.sched], self.warmup_steps, self.total_steps,
                        self.grad_accum, self.micro_batch, self.seq_len, self.seed, 1 if self.full_finetune else 0, 0)


def module_path(target: str) -> str:
    """Path of a LoRA target module inside a decoder layer: "mlp.gate_proj", "self_attn.q_proj"."""
    return f"mlp.{target}" if target in MLP_TARGETS else f"self_attn.{target}"


def linear_dims(model: ModelConfig, target: str) -> Tuple[int, int]:
    """(in, out) features of a decoder layer's linear module."""
    d, F = model.hidden, model.ffn
    dkv = (model.n_kv_heads or model.n_heads) * model.head_dim
    return {"q_proj": (d, d), "k_proj": (d, dkv), "v_proj": (d, dkv), "o_proj": (d, d), "gate_proj": (d, F), "up_proj": (d, F),
            "down_proj": (F, d)}[target]


_NP_DTYPES = {np.dtype(np.float32): DTX_F32, np.dtype(np.float16): DTX_F16}


class Trainer:
    """One GPU rank of the native fine-tuning worker (dtx_trainer handle)."""

    def __init__(self, model: ModelConfig, train: TrainConfig, device: int = 0, rank: int = 0, world: int = 1,
                 nccl_id: Optional[bytes] = None):
        self.lib = load()
        self.model, self.train = model, train
        self._h = C.c_void_p()
        mc, tc = model.to_c(), train.to_c()
        if world > 1:
            preload_nccl()
        idbuf = C.create_string_buffer(nccl_id, 128) if nccl_id is not None else None
        check(self.lib.dtx_trainer_create(C.byref(mc), C.byref(tc), device, rank, world, idbuf, C.byref(self._h)))

    def close(self) -> None:
        if self._h:
            self.lib.dtx_trainer_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- weights ------------------------------------------------------------------------------
    def load_tensor(self, name: str, arr: np.ndarray, bf16_bits: bool = False) -> None:
        """arr: float32/float16 ndarray, or uint16 ndarray holding bf16 bit patterns (bf16_bits=True)."""
        arr = np.ascontiguousarray(arr)
        dt = DTX_BF16 if bf16_bits else _NP_DTYPES[arr.dtype]
        shape = (C.c_int64 * arr.ndim)(*arr.shape)
        check(self.lib.dtx_load_tensor(self._h, name.encode(), arr.ctypes.data_as(C.c_void_p), dt, shape, arr.ndim), self._h)

    def load_state_dict(self, tensors: Dict[str, np.ndarray]) -> None:
        for k, v in tensors.items():
            self.load_tensor(k, v)

    def init_random_weights(self, seed: int) -> None:
        check(self.lib.dtx_init_random_weights(self._h, seed), self._h)

    def quantize_base(self, mode: str) -> None:
        """`--quantization int4`: the decoder weights are re-stored as packed NF4 (+ fp32 absmax per 64) on the device and
        expanded per GEMM; `int8` raises DtxError (DTX_ERR_UNSUPPORTED)."""
        check(self.lib.dtx_quantize_base(self._h, {"int4": 4, "nf4": 4, "int8": 8}[mode]), self._h)

    def init_lora(self, seed: int) -> None:
        check(self.lib.dtx_init_lora(self._h, seed), self._h)

    # -- the hot path -------------------------------------------------------------------------
    def _batch_args(self, input_ids, labels, seq_lens):
        ids = np.ascontiguousarray(input_ids, dtype=np.int32)
        lab = np.ascontiguousarray(labels, dtype=np.int32)
        assert ids.ndim == 2 and ids.shape[0] == self.train.micro_batch and lab.shape == ids.shape, (ids.shape, lab.shape)
        S = ids.shape[1]
        assert S % 128 == 0 and S <= self.train.seq_len, f"batch length {S}: a multiple of 128 and <= {self.train.seq_len} expected"
        lens = None if seq_lens is None else np.ascontiguousarray(seq_lens, dtype=np.int32)
        assert lens is None or lens.shape == (self.train.micro_batch,)
        return ids, lab, lens, S

    def step(self, input_ids: np.ndarray, labels: np.ndarray, seq_lens: Optional[np.ndarray] = None,
             force_step: bool = False) -> Tuple[float, float, float, bool]:
        """One micro-batch [micro_batch, S] (S = this batch's padded length, a multiple of 128, <= seq_len); seq_lens = true
        row lengths (None: all rows full).  Returns (loss, grad_norm, lr, stepped)."""
        ids, lab, lens, S = self._batch_args(input_ids, labels, seq_lens)
        loss, gn, lr, st = C.c_float(), C.c_float(), C.c_float(), C.c_int32()
        check(self.lib.dtx_step(self._h, ids.ctypes.data_as(C.c_void_p), lab.ctypes.data_as(C.c_void_p),
                                lens.ctypes.data_as(C.c_void_p) if lens is not None else None, S, STEP_FORCE if force_step else 0,
                                C.byref(loss), C.byref(gn), C.byref(lr), C.byref(st)), self._h)
        return loss.value, gn.value, lr.value, bool(st.value)

    def step_ptr(self, ids_ptr: int, labels_ptr: int, on_device: bool, seq_lens_ptr: int = 0,
                 seq_len_batch: int = 0) -> Tuple[float, float, float, bool]:
        """Same with raw pointers (pinned host memory, or device memory when on_device)."""
        loss, gn, lr, st = C.c_float(), C.c_float(), C.c_float(), C.c_int32()
        fn = self.lib.dtx_step_device if on_device else self.lib.dtx_step
        check(fn(self._h, C.c_void_p(ids_ptr), C.c_void_p(labels_ptr), C.c_void_p(seq_lens_ptr) if seq_lens_ptr else None,
                 seq_len_batch, 0, C.byref(loss), C.byref(gn), C.byref(lr), C.byref(st)), self._h)
        return loss.value, gn.value, lr.value, bool(st.value)

    def eval_loss(self, input_ids: np.ndarray, labels: np.ndarray, seq_lens: Optional[np.ndarray] = None) -> float:
        ids, lab, lens, S = self._batch_args(input_ids, labels, seq_lens)
        out = C.c_float()
        check(self.lib.dtx_eval_loss(self._h, ids.ctypes.data_as(C.c_void_p), lab.ctypes.data_as(C.c_void_p),
                                     lens.ctypes.data_as(C.c_void_p) if lens is not None else None, S, C.byref(out), None, None),
              self._h)
        return out.value

    def eval_rows(self, input_ids: np.ndarray, labels: np.ndarray,
                  seq_lens: Optional[np.ndarray] = None) -> Tuple[np.ndarray, np.ndarray]:
        """Forward only; returns per row (summed token loss, number of valid tokens)."""
        ids, lab, lens, S = self._batch_args(input_ids, labels, seq_lens)
        out = C.c_float()
        sums = np.zeros(self.train.micro_batch, dtype=np.float32)
        cnts = np.zeros(self.train.micro_batch, dtype=np.int32)
        check(self.lib.dtx_eval_loss(self._h, ids.ctypes.data_as(C.c_void_p), lab.ctypes.data_as(C.c_void_p),
                                     lens.ctypes.data_as(C.c_void_p) if lens is not None else None, S, C.byref(out),
                                     sums.ctypes.data_as(C.c_void_p), cnts.ctypes.data_as(C.c_void_p)), self._h)
        return sums, cnts

    def allreduce_host(self, values) -> np.ndarray:
        """Sum a small float64 vector over the ranks of this trainer's communicator."""
        v = np.ascontiguousarray(values, dtype=np.float64)
        check(self.lib.dtx_allreduce_host(self._h, v.ctypes.data_as(C.c_void_p), int(v.size)), self._h)
        return v

    # -- export -------------------------------------------------------------------------------
    def adapter_names(self) -> Iterable[str]:
        for l in range(self.model.n_layers):
            for t in self.train.lora_target:
                for ab in ("lora_A", "lora_B"):
                    yield f"base_model.model.model.layers.{l}.{module_path(t)}.{ab}.weight"

    def adapter_shape(self, name: str) -> Tuple[int, int]:
        """peft's shape of an adapter tensor: lora_A [r, in], lora_B [out, r]."""
        d_in, d_out = linear_dims(self.model, name.split(".lora_")[0].rsplit(".", 1)[-1])
        return (self.train.lora_r, d_in) if "lora_A" in name else (d_out, self.train.lora_r)

    def export_adapter(self, grads: bool = False) -> Dict[str, np.ndarray]:
        """PEFT state dict (fp32): lora_A [r, in], lora_B [out, r] per target module.  grads=True returns, under the same
        names, the summed gradient the last optimizer step consumed."""
        out = {}
        fn = self.lib.dtx_export_adapter_grad if grads else self.lib.dtx_export_adapter
        for name in self.adapter_names():
            buf = np.empty(self.adapter_shape(name), dtype=np.float32)
            check(fn(self._h, name.encode(), buf.ctypes.data_as(C.c_void_p), buf.nbytes), self._h)
            out[name] = buf
        return out

    def weight_names(self) -> Iterable[Tuple[str, Tuple[int, ...]]]:
        """(HF name, shape) of every tensor of the model, in checkpoint order."""
        m = self.model
        d, F, V, dkv = m.hidden, m.ffn, m.vocab, (m.n_kv_heads or m.n_heads) * m.head_dim
        yield "model.embed_tokens.weight", (V, d)
        for l in range(m.n_layers):
            p = f"model.layers.{l}."
            yield p + "self_attn.q_proj.weight", (d, d)
            yield p + "self_attn.k_proj.weight", (dkv, d)
            yield p + "self_attn.v_proj.weight", (dkv, d)
            yield p + "self_attn.o_proj.weight", (d, d)
            yield p + "mlp.gate_proj.weight", (F, d)
            yield p + "mlp.up_proj.weight", (F, d)
            yield p + "mlp.down_proj.weight", (d, F)
            yield p + "input_layernorm.weight", (d,)
            yield p + "post_attention_layernorm.weight", (d,)
        yield "model.norm.weight", (d,)
        yield "lm_head.weight", (V, d)

    def export_weights(self, grads: bool = False) -> Dict[str, np.ndarray]:
        """Full-parameter SFT: every weight (or its accumulated gradient) as uint16 bf16 bit patterns, HF names and layout."""
        out = {}
        for name, shape in self.weight_names():
            buf = np.empty(shape, dtype=np.uint16)
            check(self.lib.dtx_export_weight(self._h, name.encode(), buf.ctypes.data_as(C.c_void_p), buf.nbytes, 1 if grads else 0), self._h)
            out[name] = buf
        return out

    @property
    def num_trainable(self) -> int:
        return int(self.lib.dtx_num_trainable(self._h))

    @property
    def launch_count(self) -> int:
        return int(self.lib.dtx_launch_count(self._h))

    @property
    def last_step_ms(self) -> float:
        return float(self.lib.dtx_last_step_ms(self._h))

    @property
    def last_step_timings(self) -> Dict[str, float]:
        """Event-timed segments of the last step in ms."""
        out = (C.c_float * 4)()
        check(self.lib.dtx_last_step_timings(self._h, out), self._h)
        return {"step": out[0], "fwd_bwd": out[1], "allreduce": out[2], "optimizer": out[3]}

    @property
    def last_step_groups(self) -> int:
        """How the last training micro-batch was run: 0 = packed, 1 = one pass at the padded shape, > 1 = that many length groups."""
        return int(self.lib.dtx_last_step_groups(self._h))

    @property
    def base_weight_bytes(self) -> int:
        return int(self.lib.dtx_base_weight_bytes(self._h))


_nccl_preloaded = False


def preload_nccl() -> Optional[str]:
    """libdtxtune dlopen()s "libnccl.so.2" by soname.  A Python host that later imports PyTorch (the tokenizer does) needs the
    NCCL its wheel bundles (nvidia/nccl/lib/libnccl.so.2, newer than the system copy): the dynamic loader keeps ONE object per
    soname, so whichever copy is loaded first serves both.  Loading the newest copy first keeps the process consistent."""
    global _nccl_preloaded
    if _nccl_preloaded:
        return None
    _nccl_preloaded = True
    import sys
    for base in sys.path:
        cand = os.path.join(base, "nvidia", "nccl", "lib", "libnccl.so.2")
        if os.path.exists(cand):
            try:
                C.CDLL(cand, mode=C.RTLD_GLOBAL)
                return cand
            except OSError:
                pass
    return None


def nccl_unique_id() -> bytes:
    preload_nccl()
    buf = C.create_string_buffer(128)
    check(load().dtx_get_nccl_unique_id(buf))
    return buf.raw
