"""Real checkpoints and tokenizer files for the local engine.

The benchmark and the parity tests run on seeded synthetic weights and vocabularies because
nothing else exists offline (SURVEY.md §7).  With a Hugging Face model directory on disk the
same engine serves the real model:

    eng = load_pretrained("/models/Qwen3-4B", device=0)          # LocalEngine
    so  = Sutro(model_paths={"qwen-3-4b": "/models/Qwen3-4B"})    # through the SDK

What is read: `config.json` (architecture → ModelSpec), `tokenizer.json` (byte-level BPE
vocabulary, merges, special tokens), `*.safetensors` (+ `model.safetensors.index.json` when
sharded).  Supported architectures are the ones the kernels cover: Qwen3 and Llama-3 dense
decoders with head_dim 128 and a GQA group of 1, 2, 4, 5 or 8 (5: Qwen3-14B, 40 q / 8 kv heads).

Token ids.  The GPU tokenizer starts from raw byte values, so the engine's id space has byte b
at id b.  GPT-2-style vocabularies keep the 256 byte tokens at ids 0..255 in another order;
`load_tokenizer_json` therefore returns the vocabulary in ENGINE ids — the real ids with those
256 entries permuted — plus `id_map` (engine id → real id), and `load_hf_weights` callers pass
`id_map` to `pack_for_engine`, which gathers the embedding / lm_head rows accordingly.  After
that nothing on the device knows about the permutation; token ids handed back to the caller
(`return_tokens`) are engine ids and `Vocab.to_real_ids` converts them.
"""
from __future__ import annotations

import glob
import json
import os
from typing import Any, Dict, List, Optional, Tuple

import numpy as np

from . import modelspec as MS
from . import vocab as VB


# --------------------------------------------------------------------------- tokenizer.json
def _unicode_to_bytes() -> Dict[str, int]:
    return {c: b for b, c in VB._bytes_to_unicode().items()}


def load_tokenizer_json(path: str, family: str, vocab_size: Optional[int] = None) -> VB.Vocab:
    """HF `tokenizer.json` (byte-level BPE) -> Vocab in engine ids (see the module docstring)."""
    with open(path, encoding="utf-8") as f:
        tj = json.load(f)
    model = tj.get("model", {})
    if model.get("type") != "BPE":
        raise ValueError(f"{path}: only byte-level BPE tokenizers are supported "
                         f"(model.type = {model.get('type')!r})")
    u2b = _unicode_to_bytes()
    digits = _pretokenizer_digits(tj.get("pre_tokenizer"), path)
    if digits is None:
        digits = 1 if family == "qwen3" else 3
    norm = tj.get("normalizer")
    if norm is not None and norm.get("type") != "NFC":
        raise ValueError(f"{path}: normalizer {norm.get('type')!r} is not supported (NFC or none)")

    def to_bytes(tok: str) -> bytes:
        try:
            return bytes(u2b[c] for c in tok)
        except KeyError:
            raise ValueError(f"{path}: token {tok!r} is not byte-level encoded") from None

    real_vocab: Dict[str, int] = model["vocab"]
    added = {a["content"]: int(a["id"]) for a in tj.get("added_tokens", [])}
    n_ids = max(max(real_vocab.values(), default=-1), max(added.values(), default=-1)) + 1
    size = max(n_ids, vocab_size or 0)
    real_bytes: List[bytes] = [b""] * size
    for tok, i in real_vocab.items():
        if tok in added:
            continue
        real_bytes[i] = to_bytes(tok)
    byte_id = [-1] * 256
    for i, tb in enumerate(real_bytes[:n_ids]):
        if len(tb) == 1 and byte_id[tb[0]] < 0:
            byte_id[tb[0]] = i
    if sorted(byte_id) != list(range(256)):
        raise ValueError(f"{path}: the 256 byte tokens do not occupy ids 0..255 — this "
                         "vocabulary layout is not supported")
    e2r = np.arange(size, dtype=np.int32)
    e2r[:256] = np.asarray(byte_id, dtype=np.int32)
    r2e = np.empty(size, dtype=np.int32)
    r2e[e2r] = np.arange(size, dtype=np.int32)
    token_bytes = [real_bytes[int(e2r[e])] for e in range(size)]

    merges: List[Tuple[int, int]] = []
    merged_ids: List[int] = []
    for m in model.get("merges", []):
        a, b = m.split(" ") if isinstance(m, str) else m
        ab = a + b
        if a not in real_vocab or b not in real_vocab or ab not in real_vocab:
            continue          # a merge whose parts or result are not tokens can never apply
        merges.append((int(r2e[real_vocab[a]]), int(r2e[real_vocab[b]])))
        merged_ids.append(int(r2e[real_vocab[ab]]))
    word_overrides = None
    if model.get("ignore_merges"):
        # `ignore_merges` (Llama-3 files set it): a pre-token that is itself in the vocabulary
        # is emitted as that token without running the merges.  That differs from plain BPE only
        # for entries whose merges build something else: list those, with the sequence their
        # merges do build — the GPU tokenizer replaces exactly those sequences (two byte strings
        # never merge to the same tokens, so the replacement is exact).
        rank = {pair: (i, merged_ids[i]) for i, pair in reversed(list(enumerate(merges)))}
        word_overrides = []
        for e, tb in enumerate(token_bytes):
            if len(tb) < 2:
                continue
            seq = list(tb)
            while len(seq) > 1:
                best, bi = None, -1
                for i in range(len(seq) - 1):
                    r = rank.get((seq[i], seq[i + 1]))
                    if r is not None and (best is None or r[0] < best[0]):
                        best, bi = r, i
                if best is None:
                    break
                seq[bi:bi + 2] = [best[1]]
            if len(seq) >= 2:
                if len(seq) > 32:
                    raise ValueError(
                        f"{path}: model.ignore_merges is true and vocabulary entry {e} merges to "
                        f"{len(seq)} tokens; the GPU tokenizer's whole-word table holds sequences "
                        "of at most 32")
                word_overrides.append((tuple(seq), e))
    specials = {name: int(r2e[i]) for name, i in added.items()}
    need = "<|im_end|>" if family == "qwen3" else "<|eot_id|>"
    if need not in specials:
        raise ValueError(f"{path}: special token {need!r} (end of turn) is missing")
    return VB.Vocab(family, size, token_bytes, merges, specials, digits,
                    merged_ids=merged_ids, id_map=e2r, normalize_nfc=norm is not None,
                    word_overrides=word_overrides)


def _pretokenizer_digits(pre: Optional[Dict[str, Any]], path: str) -> Optional[int]:
    """The GPU pre-tokeniser implements one pattern family (vocab.PRETOK_PATTERN, numbers in runs
    of 1 or 3 digits).  Returns the digit run length the file asks for, None when the file does
    not say, and raises when it asks for a different pattern."""
    if pre is None:
        return None
    steps = pre.get("pretokenizers", [pre])
    for step in steps:
        if step.get("type") == "Split":
            rx = step.get("pattern", {}).get("Regex")
            for d in (1, 3):
                ours = VB.PRETOK_PATTERN % d
                if rx in (ours, ours.replace("\\p{N}{1,1}", "\\p{N}")):
                    return d
            raise ValueError(f"{path}: pre-tokeniser pattern {rx!r} is not the GPT-4-style pattern "
                             "the GPU tokenizer implements")
        if step.get("type") not in ("ByteLevel", "Sequence"):
            raise ValueError(f"{path}: pre-tokeniser step {step.get('type')!r} is not supported")
    return None


# --------------------------------------------------------------------------- config.json
def spec_from_hf_config(cfg: Dict[str, Any], name: str, max_position: int = 4096,
                        embedding_model: bool = False) -> MS.ModelSpec:
    mt = cfg.get("model_type")
    if mt not in ("qwen3", "llama"):
        raise ValueError(f"unsupported model_type {mt!r}: the kernels cover Qwen3 and Llama-3 "
                         "dense decoders")
    d_model, hq = int(cfg["hidden_size"]), int(cfg["num_attention_heads"])
    hkv = int(cfg.get("num_key_value_heads", hq))
    head_dim = int(cfg.get("head_dim") or d_model // hq)
    if head_dim != MS.HEAD_DIM:
        raise ValueError(f"head_dim {head_dim} is not supported (kernels are built for "
                         f"{MS.HEAD_DIM})")
    if hq % hkv or hq // hkv not in (1, 2, 4, 5, 8):
        raise ValueError(f"GQA group {hq}/{hkv} is not supported (1, 2, 4, 5 or 8)")
    if cfg.get("attention_bias") or cfg.get("mlp_bias"):
        raise ValueError("projection biases are not supported")
    if cfg.get("sliding_window") and cfg.get("use_sliding_window"):
        raise ValueError("sliding-window attention is not supported")
    # transformers >= 5 writes rope_theta (and any scaling) under rope_parameters
    rope_params = cfg.get("rope_parameters") or {}
    theta = cfg.get("rope_theta") or rope_params.get("rope_theta", 1e4)
    scaling = cfg.get("rope_scaling")
    if scaling is None and rope_params.get("rope_type", "default") != "default":
        scaling = rope_params
    if scaling is not None:
        kind = scaling.get("rope_type", scaling.get("type"))
        if kind != "llama3":
            raise ValueError(f"rope scaling {kind!r} is not supported")
        scaling = {k: scaling[k] for k in ("factor", "low_freq_factor", "high_freq_factor",
                                           "original_max_position_embeddings")}
    return MS.ModelSpec(
        name=name, family="qwen3" if mt == "qwen3" else "llama",
        n_layers=int(cfg["num_hidden_layers"]), d_model=d_model, n_q_heads=hq, n_kv_heads=hkv,
        d_ff=int(cfg["intermediate_size"]), vocab_size=int(cfg["vocab_size"]),
        tied_embeddings=bool(cfg.get("tie_word_embeddings", False)),
        rms_eps=float(cfg.get("rms_norm_eps", 1e-6)), rope_theta=float(theta),
        qk_norm=(mt == "qwen3"),
        max_position=min(int(cfg.get("max_position_embeddings", max_position)), max_position),
        rope_scaling=scaling, embedding_model=embedding_model)


# --------------------------------------------------------------------------- safetensors
def load_hf_weights(model_dir: str) -> Dict[str, "Any"]:
    """Every tensor of the checkpoint, bf16, HF names (`model.layers.N...`, `lm_head.weight`)."""
    import torch
    from safetensors import safe_open
    files = sorted(glob.glob(os.path.join(model_dir, "*.safetensors")))
    index = os.path.join(model_dir, "model.safetensors.index.json")
    if os.path.exists(index):
        with open(index) as f:
            files = sorted({os.path.join(model_dir, x) for x in json.load(f)["weight_map"].values()})
    if not files:
        raise FileNotFoundError(f"no *.safetensors files in {model_dir}")
    out: Dict[str, Any] = {}
    for fn in files:
        with safe_open(fn, framework="pt", device="cpu") as f:
            for k in f.keys():
                t = f.get_tensor(k)
                out[k if k.startswith(("model.", "lm_head.")) else "model." + k] = \
                    t.to(torch.bfloat16)
    return out


def load_pretrained(model_dir: str, device=0, name: Optional[str] = None,
                    max_position: int = 4096, embedding_model: Optional[bool] = None, **engine_kw):
    """-> LocalEngine serving the checkpoint in `model_dir`."""
    from .engine import LocalEngine
    with open(os.path.join(model_dir, "config.json")) as f:
        cfg = json.load(f)
    name = name or os.path.basename(os.path.normpath(model_dir))
    if embedding_model is None:
        embedding_model = "embedding" in name.lower()
    spec = spec_from_hf_config(cfg, name, max_position, embedding_model)
    v = load_tokenizer_json(os.path.join(model_dir, "tokenizer.json"), spec.family,
                            spec.vocab_size)
    if v.vocab_size != spec.vocab_size:
        raise ValueError(f"tokenizer has ids up to {v.vocab_size - 1} but the model has "
                         f"{spec.vocab_size} embedding rows")
    w = load_hf_weights(model_dir)
    ew = MS.pack_for_engine(spec, w, device if isinstance(device, str) else f"cuda:{device}",
                            row_map=v.id_map)
    eng = LocalEngine(spec, ew, v, device=device, **engine_kw)
    # released Qwen3 chat models answer directly only when the turn opens with an empty think block
    eng.empty_think_block = (spec.family == "qwen3" and not spec.embedding_model
                             and "thinking" not in name.lower())
    return eng
