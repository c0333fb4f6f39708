"""Model architecture specs and seeded synthetic weights.

The reference names models but ships none (sutro/common.py:11-45 is a list of
strings forwarded to the hosted service).  The architectures here are the public
model-card values for the names BASELINE.json uses; no checkpoint exists offline
so weights are random-initialised from a seed (stated in every report).

One spec feeds both the CPU oracle (oracle/model_ref.py, HF-style tensor names)
and the engine (fused/interleaved layouts built by `pack_for_engine`).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field, replace
from typing import Dict, Optional

import numpy as np
import torch

HEAD_DIM = 128  # every supported architecture uses 128-wide heads (kernels assume it)


@dataclass(frozen=True)
class ModelSpec:
    name: str
    family: str            # "qwen3" | "llama"
    n_layers: int
    d_model: int
    n_q_heads: int
    n_kv_heads: int
    d_ff: int
    vocab_size: int
    tied_embeddings: bool
    rms_eps: float
    rope_theta: float
    qk_norm: bool
    max_position: int = 4096          # context window the engine serves (truncate_rows bound)
    rope_scaling: Optional[dict] = None  # llama3-style {"factor","low_freq_factor",...}
    embedding_model: bool = False     # prefill-only, last-token pool + L2 normalise
    head_dim: int = HEAD_DIM

    @property
    def q_dim(self) -> int:
        return self.n_q_heads * self.head_dim

    @property
    def kv_dim(self) -> int:
        return self.n_kv_heads * self.head_dim

    @property
    def qkv_dim(self) -> int:
        return self.q_dim + 2 * self.kv_dim

    @property
    def kv_bytes_per_token(self) -> int:
        return 2 * self.n_layers * self.n_kv_heads * self.head_dim * 2

    def n_params(self) -> int:
        per_layer = (self.qkv_dim * self.d_model + self.d_model * self.q_dim +
                     3 * self.d_ff * self.d_model + 2 * self.d_model +
                     (2 * self.head_dim if self.qk_norm else 0))
        emb = self.vocab_size * self.d_model
        return self.n_layers * per_layer + emb * (1 if self.tied_embeddings else 2) + self.d_model

    def matmul_flops_per_token(self, with_lm_head: bool = True) -> int:
        per_layer = 2 * (self.qkv_dim * self.d_model + self.d_model * self.q_dim +
                         3 * self.d_ff * self.d_model)
        f = self.n_layers * per_layer
        if with_lm_head:
            f += 2 * self.vocab_size * self.d_model
        return f


_LLAMA31_SCALING = {"factor": 8.0, "low_freq_factor": 1.0, "high_freq_factor": 4.0,
                    "original_max_position_embeddings": 8192}

SPECS: Dict[str, ModelSpec] = {}


def _reg(s: ModelSpec) -> ModelSpec:
    SPECS[s.name] = s
    return s


QWEN3_0_6B = _reg(ModelSpec("qwen-3-0.6b", "qwen3", 28, 1024, 16, 8, 3072, 151936, True, 1e-6,
                            1e6, True))
QWEN3_EMB_0_6B = _reg(replace(QWEN3_0_6B, name="qwen-3-embedding-0.6b", embedding_model=True))
QWEN3_4B = _reg(ModelSpec("qwen-3-4b", "qwen3", 36, 2560, 32, 8, 9728, 151936, True, 1e-6, 1e6,
                          True))
# GQA group 5 (40 q / 8 kv heads): the attention kernels' only non-power-of-two group
QWEN3_14B = _reg(ModelSpec("qwen-3-14b", "qwen3", 40, 5120, 40, 8, 17408, 151936, False, 1e-6,
                           1e6, True))
QWEN3_32B = _reg(ModelSpec("qwen-3-32b", "qwen3", 64, 5120, 64, 8, 25600, 151936, False, 1e-6,
                           1e6, True))
LLAMA31_8B = _reg(ModelSpec("llama-3.1-8b", "llama", 32, 4096, 32, 8, 14336, 128256, False, 1e-5,
                            5e5, False, rope_scaling=_LLAMA31_SCALING))
# BASELINE.json says "llama-3-8b"; the reference's ModelOptions lists llama-3.1-8b
# (sutro/common.py:22).  Same shapes; alias it.
SPECS["llama-3-8b"] = LLAMA31_8B
SPECS["qwen-3-0.6B"] = QWEN3_0_6B

# Tiny architectures for parity tests (same code paths, seconds on CPU).
TINY_QWEN3 = _reg(ModelSpec("tiny-qwen3", "qwen3", 2, 256, 4, 2, 512, 1024, True, 1e-6, 1e6, True,
                            max_position=512))
TINY_QWEN3_G4 = _reg(ModelSpec("tiny-qwen3-g4", "qwen3", 3, 512, 8, 2, 768, 2048, True, 1e-6, 1e6,
                               True, max_position=1024))
TINY_QWEN3_G5 = _reg(ModelSpec("tiny-qwen3-g5", "qwen3", 3, 512, 10, 2, 768, 2048, True, 1e-6,
                               1e6, True, max_position=1024))
TINY_LLAMA = _reg(ModelSpec("tiny-llama", "llama", 2, 256, 4, 2, 512, 1024, False, 1e-5, 5e5,
                            False, max_position=512, rope_scaling=_LLAMA31_SCALING))
TINY_EMB = _reg(replace(TINY_QWEN3, name="tiny-qwen3-embedding", embedding_model=True))


def get_spec(name: str) -> ModelSpec:
    if name in SPECS:
        return SPECS[name]
    base = name.replace("-thinking", "")
    if base in SPECS:
        return SPECS[base]
    raise ValueError(f"Unknown model '{name}'. Local engine supports: {sorted(SPECS)}")


def with_vocab(spec: ModelSpec, vocab_size: int) -> ModelSpec:
    return replace(spec, vocab_size=vocab_size)


# --------------------------------------------------------------------------- RoPE tables
def rope_inv_freq(spec: ModelSpec) -> torch.Tensor:
    """fp32 inverse frequencies, restating transformers 5.5.0 modeling_rope_utils.py
    (default: :130-160, llama3: :550-600)."""
    hd = spec.head_dim
    inv = 1.0 / (spec.rope_theta ** (torch.arange(0, hd, 2, dtype=torch.int64).float() / hd))
    sc = spec.rope_scaling
    if sc:
        factor, lo, hi = sc["factor"], sc["low_freq_factor"], sc["high_freq_factor"]
        old = sc["original_max_position_embeddings"]
        low_wl, high_wl = old / lo, old / hi
        wavelen = 2 * math.pi / inv
        inv_llama = torch.where(wavelen > low_wl, inv / factor, inv)
        smooth = (old / wavelen - lo) / (hi - lo)
        smoothed = (1 - smooth) * inv_llama / factor + smooth * inv_llama
        is_medium = ~(wavelen < high_wl) * ~(wavelen > low_wl)
        inv = torch.where(is_medium, smoothed, inv_llama)
    return inv


def rope_tables(spec: ModelSpec, max_pos: Optional[int] = None):
    """(cos, sin) as bf16 [max_pos, head_dim/2] — computed in fp32 then rounded to the
    model dtype exactly as the reference model does before applying them."""
    n = max_pos or spec.max_position
    inv = rope_inv_freq(spec)
    freqs = torch.arange(n, dtype=torch.float32)[:, None] * inv[None, :]
    return freqs.cos().to(torch.bfloat16), freqs.sin().to(torch.bfloat16)


# --------------------------------------------------------------------------- weights
def make_weights(spec: ModelSpec, seed: int = 0, device: str = "cpu",
                 std: float = 0.02) -> Dict[str, torch.Tensor]:
    """Seeded random weights, bf16, HF tensor names.  Norm weights are 1 + small noise so
    that the multiply is actually exercised."""
    g = torch.Generator(device=device).manual_seed(seed)

    def rnd(*shape, s=std):
        return (torch.randn(*shape, generator=g, device=device, dtype=torch.float32) * s).to(
            torch.bfloat16)

    def norm(n):
        return (1.0 + torch.randn(n, generator=g, device=device, dtype=torch.float32) * 0.1).to(
            torch.bfloat16)

    w: Dict[str, torch.Tensor] = {}
    w["model.embed_tokens.weight"] = rnd(spec.vocab_size, spec.d_model)
    for i in range(spec.n_layers):
        p = f"model.layers.{i}."
        w[p + "input_layernorm.weight"] = norm(spec.d_model)
        w[p + "self_attn.q_proj.weight"] = rnd(spec.q_dim, spec.d_model)
        w[p + "self_attn.k_proj.weight"] = rnd(spec.kv_dim, spec.d_model)
        w[p + "self_attn.v_proj.weight"] = rnd(spec.kv_dim, spec.d_model)
        w[p + "self_attn.o_proj.weight"] = rnd(spec.d_model, spec.q_dim)
        if spec.qk_norm:
            w[p + "self_attn.q_norm.weight"] = norm(spec.head_dim)
            w[p + "self_attn.k_norm.weight"] = norm(spec.head_dim)
        w[p + "post_attention_layernorm.weight"] = norm(spec.d_model)
        w[p + "mlp.gate_proj.weight"] = rnd(spec.d_ff, spec.d_model)
        w[p + "mlp.up_proj.weight"] = rnd(spec.d_ff, spec.d_model)
        w[p + "mlp.down_proj.weight"] = rnd(spec.d_model, spec.d_ff)
    w["model.norm.weight"] = norm(spec.d_model)
    if not spec.tied_embeddings:
        w["lm_head.weight"] = rnd(spec.vocab_size, spec.d_model)
    return w


@dataclass
class EngineWeights:
    """Device tensors in the layouts the kernels want (all bf16, contiguous)."""
    embed: torch.Tensor                 # [V, d]
    lm_head: torch.Tensor               # [V, d] (aliases embed when tied)
    final_norm: torch.Tensor            # [d]
    ln1: list = field(default_factory=list)       # per layer [d]
    ln2: list = field(default_factory=list)
    wqkv: list = field(default_factory=list)      # [qkv_dim, d]   rows: q | k | v
    wo: list = field(default_factory=list)        # [d, q_dim]
    wgu: list = field(default_factory=list)       # [2*d_ff, d]    rows interleaved gate,up
    wd: list = field(default_factory=list)        # [d, d_ff]
    q_norm: list = field(default_factory=list)    # [128] or None
    k_norm: list = field(default_factory=list)

    def all_tensors(self):
        seen, out = set(), []
        for t in [self.embed, self.lm_head, self.final_norm, *self.ln1, *self.ln2, *self.wqkv,
                  *self.wo, *self.wgu, *self.wd, *self.q_norm, *self.k_norm]:
            if t is not None and t.data_ptr() not in seen:
                seen.add(t.data_ptr())
                out.append(t)
        return out


def pack_for_engine(spec: ModelSpec, w: Dict[str, torch.Tensor], device,
                    row_map=None) -> EngineWeights:
    """HF-named tensors -> engine layout on `device`.  `row_map` (engine id -> checkpoint id,
    `Vocab.id_map` of a real tokenizer file) reorders the embedding / lm_head rows."""
    dev = torch.device(device)

    def d(t):
        return t.to(dev).contiguous()

    def rows(t):
        if row_map is None:
            return d(t)
        return d(t[torch.as_tensor(np.asarray(row_map), dtype=torch.long)])

    embed = rows(w["model.embed_tokens.weight"])
    ew = EngineWeights(embed=embed,
                       lm_head=embed if spec.tied_embeddings else rows(w["lm_head.weight"]),
                       final_norm=d(w["model.norm.weight"]))
    for i in range(spec.n_layers):
        p = f"model.layers.{i}."
        ew.ln1.append(d(w[p + "input_layernorm.weight"]))
        ew.ln2.append(d(w[p + "post_attention_layernorm.weight"]))
        ew.wqkv.append(d(torch.cat([w[p + "self_attn.q_proj.weight"],
                                    w[p + "self_attn.k_proj.weight"],
                                    w[p + "self_attn.v_proj.weight"]], dim=0)))
        ew.wo.append(d(w[p + "self_attn.o_proj.weight"]))
        gu = torch.stack([w[p + "mlp.gate_proj.weight"], w[p + "mlp.up_proj.weight"]], dim=1)
        ew.wgu.append(d(gu.reshape(2 * spec.d_ff, spec.d_model)))
        ew.wd.append(d(w[p + "mlp.down_proj.weight"]))
        ew.q_norm.append(d(w[p + "self_attn.q_norm.weight"]) if spec.qk_norm else None)
        ew.k_norm.append(d(w[p + "self_attn.k_norm.weight"]) if spec.qk_norm else None)
    return ew


def make_engine_weights_on_device(spec: ModelSpec, seed: int, device) -> EngineWeights:
    """Generate directly in engine layout on the GPU (bench path: 8 GB of weights
    would take minutes to draw on the host).  Layer by layer to bound peak memory."""
    dev = torch.device(device)
    g = torch.Generator(device=dev).manual_seed(seed)

    def rnd(*shape):
        return (torch.randn(*shape, generator=g, device=dev, dtype=torch.float32) * 0.02).to(
            torch.bfloat16)

    def norm(n):
        return (1.0 + torch.randn(n, generator=g, device=dev, dtype=torch.float32) * 0.1).to(
            torch.bfloat16)

    embed = rnd(spec.vocab_size, spec.d_model)
    ew = EngineWeights(embed=embed,
                       lm_head=embed if spec.tied_embeddings else rnd(spec.vocab_size,
                                                                     spec.d_model),
                       final_norm=norm(spec.d_model))
    for _ in range(spec.n_layers):
        ew.ln1.append(norm(spec.d_model))
        ew.ln2.append(norm(spec.d_model))
        ew.wqkv.append(rnd(spec.qkv_dim, spec.d_model))
        ew.wo.append(rnd(spec.d_model, spec.q_dim))
        ew.wgu.append(rnd(2 * spec.d_ff, spec.d_model))
        ew.wd.append(rnd(spec.d_model, spec.d_ff))
        ew.q_norm.append(norm(spec.head_dim) if spec.qk_norm else None)
        ew.k_norm.append(norm(spec.head_dim) if spec.qk_norm else None)
    return ew


def unpack_to_hf(spec: ModelSpec, ew: EngineWeights) -> Dict[str, torch.Tensor]:
    """Inverse of pack_for_engine (CPU copies, HF names) — lets the CPU baseline run on
    the very weights the engine generated on the GPU."""
    w: Dict[str, torch.Tensor] = {"model.embed_tokens.weight": ew.embed.cpu(),
                                  "model.norm.weight": ew.final_norm.cpu()}
    if not spec.tied_embeddings:
        w["lm_head.weight"] = ew.lm_head.cpu()
    for i in range(spec.n_layers):
        p = f"model.layers.{i}."
        qkv = ew.wqkv[i].cpu()
        w[p + "self_attn.q_proj.weight"] = qkv[:spec.q_dim]
        w[p + "self_attn.k_proj.weight"] = qkv[spec.q_dim:spec.q_dim + spec.kv_dim]
        w[p + "self_attn.v_proj.weight"] = qkv[spec.q_dim + spec.kv_dim:]
        w[p + "self_attn.o_proj.weight"] = ew.wo[i].cpu()
        gu = ew.wgu[i].cpu().view(spec.d_ff, 2, spec.d_model)
        w[p + "mlp.gate_proj.weight"] = gu[:, 0].contiguous()
        w[p + "mlp.up_proj.weight"] = gu[:, 1].contiguous()
        w[p + "mlp.down_proj.weight"] = ew.wd[i].cpu()
        w[p + "input_layernorm.weight"] = ew.ln1[i].cpu()
        w[p + "post_attention_layernorm.weight"] = ew.ln2[i].cpu()
        if spec.qk_norm:
            w[p + "self_attn.q_norm.weight"] = ew.q_norm[i].cpu()
            w[p + "self_attn.k_norm.weight"] = ew.k_norm[i].cpu()
    return w
