#!/usr/bin/env python
"""Benchmark of the so.infer() hot path (BASELINE.json metric: rows/s and output tok/s over a
DataFrame column at 1/2/4/8 B200; % of roofline for the dominant kernels).

    python bench.py --gpus 1 --steps 3 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference            # CPU baseline arm

Workload (config.workload): BASELINE.json configs[1] — ONE 20k-row synthetic product-review
frame per step, qwen-3-4b architecture in bf16 (seeded random weights: no checkpoint exists
offline), system prompt + Sentiment enum output_schema, greedy.  The frame lives on rank 0.

One "step" = one call of the public API on that frame, exactly what a user runs:

    so.infer(df, column="review_text", model="qwen-3-4b", system_prompt=..., output_schema=...)

  N = 1   the SDK hands the column to `sb200_infer_text` — one C-ABI call, host buffers in and out.
  N > 1   every rank makes the same call (one process per GPU, torchrun); the SDK takes the
          row-sharded path (sutro_b200/sharding.py `infer_frame_sharded`): rank 0's column goes to
          HBM, NCCL broadcast, every rank selects its length-balanced share with a native
          kernel, runs it on its replica, NCCL gather on rank 0, ordered merge (results are
          positional, sutro/sdk.py:406-412), device -> host, write-back into the frame.
          STRONG scaling: the same 20k rows at every N.

`e2e`    = rows/s of the K calls: barrier + synchronize on both sides, wall clock, host frame in,
           result column written back — host<->device copies inside.
`value`  = rows/s with the inputs already resident in HBM: CUDA-event time from "column resident
           in (rank 0's) HBM" to "ordered results resident in (rank 0's) HBM" — at N>1 that
           includes the broadcast, the slowest rank and the gather.
Secondary blocks (N = 1 only, after the timed region, bounded samples): configs[2] (512-token
documents, 64 generated tokens, no schema: the decode-attention-heavy regime), configs[3]
(qwen-3-embedding-0.6b, prefill only) and configs[4] (llama-3.1-8b, nested output_schema).
The reference arm (`--impl reference`) times the CPU oracle — there is no reference CPU
implementation of this path to time (SURVEY.md §0); it is labelled "port".
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SYSTEM_PROMPT = "Classify the sentiment of the review as positive, neutral, or negative."
SCHEMA = {"type": "object", "title": "Sentiment",
          "properties": {"sentiment": {"type": "string",
                                       "enum": ["positive", "neutral", "negative"]}},
          "required": ["sentiment"]}
MAX_NEW = 24
COLUMN = "review_text"          # the README's column name (README.md:72)

# configs[4]: nested output_schema (object -> list of objects -> {str, int(min,max), enum,
# optional float}); written as JSON Schema so that bench.py needs no pydantic at import time
ORDER_SCHEMA = {
    "$defs": {"Item": {"type": "object", "title": "Item", "properties": {
        "name": {"type": "string", "maxLength": 12},
        "quantity": {"type": "integer", "minimum": 0, "maximum": 1000},
        "kind": {"type": "string", "enum": ["a", "b", "c"]},
        "price": {"anyOf": [{"type": "number"}, {"type": "null"}], "default": None}},
        "required": ["name", "quantity", "kind"]}},
    "type": "object", "title": "Order",
    "properties": {"customer": {"type": "string", "maxLength": 10},
                   "items": {"type": "array", "items": {"$ref": "#/$defs/Item"}, "maxItems": 3},
                   "paid": {"type": "boolean"}},
    "required": ["customer", "items", "paid"]}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0,
            "source": "fallback"}


def ncu_traffic(csv_name: str, kernel: str):
    """DRAM bytes (read + write) of one launch of `kernel` (substring of the kernel name) from a
    committed `ncu --set full` capture under profiles/ (the per-launch summary
    tools/profile_extract.py writes), or None.  The capture is of one representative launch of
    the kernel class inside the same workload, not of this run."""
    try:
        import csv
        with open(os.path.join(ROOT, "profiles", csv_name), newline="") as f:
            rows = list(csv.reader(f))
        hdr = rows[0]
        scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        cols = []
        for i, h in enumerate(hdr):
            if h.startswith(("dram_read", "dram_write")):
                cols.append((i, scale[h[h.index("[") + 1:h.index("]")]]))
        for r in rows[1:]:
            if kernel in r[0]:
                return sum(float(r[i]) * k for i, k in cols)
        return None
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled during the timed region."""

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                 str(self.idx), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names)
                   if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        loaded = sorted(sm)[len(sm) // 4:]  # drop idle samples between steps
        return {"sm_mhz": statistics.median(loaded), "sm_max_mhz": float(self.rows[0][1]),
                "reasons": reasons, "samples": len(sm),
                "power_w_max": max(float(r[2]) for r in self.rows if len(r) >= 7)}


_T0 = time.perf_counter()


def log(msg: str):
    """progress to stderr (stdout carries exactly one JSON line)"""
    if int(os.environ.get("RANK", "0")) == 0:
        print(f"[bench +{time.perf_counter() - _T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


# stdout must carry exactly one JSON line: libraries that print there (NCCL's version
# banner) are diverted to stderr for the life of the process; emit() writes to the real fd.
_REAL_STDOUT = None


def divert_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


WORKLOAD = "sentiment"   # set from --workload


def make_rows(n: int, seed: int):
    from sutro_b200 import synth
    if WORKLOAD == "docs":   # BASELINE.json configs[2]: ~512-token prompts, 64 generated, no schema
        return synth.documents(n, seed=seed, words=475)
    return synth.product_reviews(n, seed=seed)


def infer_kwargs(model: str):
    """Arguments of the public call for the selected workload."""
    if WORKLOAD == "docs":
        return dict(model=model, column=COLUMN,
                    sampling_params={"max_tokens": 64, "ignore_eos": True})
    return dict(model=model, column=COLUMN, system_prompt=SYSTEM_PROMPT, output_schema=SCHEMA,
                sampling_params={"max_tokens": MAX_NEW})


def gen_kwargs():
    """The same job as engine-level arguments (profiled step, secondary blocks)."""
    if WORKLOAD == "docs":
        return dict(system_prompt=None, json_schema=None, max_new_tokens=64, ignore_eos=True)
    return dict(system_prompt=SYSTEM_PROMPT, json_schema=SCHEMA, max_new_tokens=MAX_NEW)


# ----------------------------------------------------------------------------- CPU arm
def cpu_baseline(spec, hf_weights, vocab, rows, threads: int, budget_s: float = 25.0):
    """Times the CPU oracle (oracle/: the checker, here only as the measured baseline) on
    a bounded sample of the same workload: rows are processed until `budget_s` of CPU work
    has been spent (at least one row).  Returns the record and the oracle's output strings."""
    import torch
    from oracle.bpe_ref import RefTokenizer
    from oracle.fsm_ref import TokenFSM
    from oracle.model_ref import RefModel
    from sutro_b200 import vocab as VB
    from sutro_b200.schema_fsm import compile_schema
    threads = max(1, min(threads, 64))   # tiny per-op kernels stop scaling long before that
    torch.set_num_threads(threads)
    t_init = time.perf_counter()
    tok, model = RefTokenizer(vocab), RefModel(spec, hf_weights, fast=True)
    fsm = TokenFSM(compile_schema(SCHEMA), vocab)
    fsm.enable_jump_forward(tok)    # same decoding algorithm as the engine (jump-forward)
    tpl = VB.chat_template(spec.family, SYSTEM_PROMPT)
    log(f"cpu baseline: oracle ready in {time.perf_counter() - t_init:.1f}s, {threads} threads")
    import signal

    class _Timeout(Exception):
        pass

    def _on_alarm(signum, frame):
        raise _Timeout()

    hard_limit = max(60.0, 6 * budget_s)       # never let the baseline sink the benchmark
    old = signal.signal(signal.SIGALRM, _on_alarm)
    signal.setitimer(signal.ITIMER_REAL, hard_limit)
    t0, n_out, n_rows, partial = time.perf_counter(), 0, 0, 0.0
    texts, min_margins = [], []
    try:
        for r in rows:
            g = model.generate(tok.render(tpl, r), MAX_NEW, vocab.eos_id, fsm=fsm)
            n_out += len(g.tokens)
            texts.append(tok.decode(g.tokens) if hasattr(tok, "decode") else None)
            min_margins.append(min(g.margins) if g.margins else None)
            n_rows += 1
            log(f"cpu baseline: row {n_rows} done at +{time.perf_counter() - t0:.1f}s")
            if time.perf_counter() - t0 > budget_s:
                break
    except _Timeout:
        log(f"cpu baseline: hard limit {hard_limit:.0f}s hit after {n_rows} complete rows")
        if n_rows == 0:
            partial = 1.0   # report an upper bound: less than one row in hard_limit seconds
    finally:
        signal.setitimer(signal.ITIMER_REAL, 0)
        signal.signal(signal.SIGALRM, old)
    dt = time.perf_counter() - t0
    if partial:
        return {"value": 1.0 / dt, "unit": "rows/s", "cores": threads, "kind": "port",
                "sample": f"UPPER BOUND: the first row did not finish within {dt:.0f} s "
                          "(oracle/model_ref.py, torch CPU)", "output_tokens_per_s": None}, [], []
    return {"value": n_rows / dt, "unit": "rows/s", "cores": threads, "kind": "port",
            "sample": f"{n_rows} rows of the same frame in {dt:.1f} s, one row at a time, "
                      "oracle/model_ref.py (torch CPU fp32 GEMM on bf16-valued weights); the "
                      "reference repo has no local implementation of this path",
            "output_tokens_per_s": n_out / dt}, texts, min_margins


DUMP_LIMIT = 64 << 20   # bytes, both --dump-outputs files together


def dump_width(vocab, max_new_tokens: int) -> int:
    """Longest result string, in code points, a job can return: at most `max_new_tokens`
    tokens (forced tokens included), decoded with errors='replace', which never yields
    more code points than bytes."""
    return max_new_tokens * max(len(b) for b in vocab.token_bytes)


def dump_outputs(dirname: str, outputs, width: int, limit: int = DUMP_LIMIT):
    """--dump-outputs: the result column of the last timed step, as the caller receives it.
    `inference_result.npy` holds row r's Unicode code points as float32 values (exact up to
    U+10FFFF), padded with -1 to `width` (dump_width); `row_index.npy` (float64) gives the
    frame row of each line.  If all rows would not fit in `limit` bytes, a fixed seeded
    sample of rows is written instead.  Width and sample follow from the row count and the
    arguments only, so two builds run with the same arguments write arrays of one shape."""
    import numpy as np
    n = len(outputs)
    keep = min(n, (limit - 4096) // (4 * width + 8))     # 4096: room for the two .npy headers
    idx = np.arange(n) if keep == n else \
        np.sort(np.random.RandomState(0).choice(n, keep, replace=False))
    arr = np.full((len(idx), width), -1.0, dtype=np.float32)
    for r, i in enumerate(idx):
        cp = np.frombuffer(outputs[i].encode("utf-32-le"), dtype="<u4")
        arr[r, :len(cp)] = cp
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "inference_result.npy"), arr)
    np.save(os.path.join(dirname, "row_index.npy"), idx.astype(np.float64))
    log(f"dumped {len(idx)}/{n} result rows to {dirname}")


def plumbing_cost(model, rows, outputs):
    """SURVEY.md §8(d): the only code of this path the reference runs locally is the host
    plumbing — column extraction (sutro/common.py:111-149), payload build + JSON encode
    (sutro/sdk.py:196-208) and positional write-back (:408-412).  Timed here through this
    repo's restatement (sutro_b200.common; pinned to the reference by tests/golden/
    plumbing.json) on the benchmark's own rows, single thread."""
    import pandas as pd
    from sutro_b200.common import handle_data_helper
    df = pd.DataFrame({COLUMN: rows})
    t0 = time.perf_counter()
    inputs = handle_data_helper(df, COLUMN)
    payload = {"model": model, "inputs": inputs, "job_priority": 0, "json_schema": None,
               "system_prompt": None, "cost_estimate": False, "sampling_params": None,
               "random_seed_per_input": False, "truncate_rows": True, "name": None,
               "description": None}
    body = json.dumps(payload)
    df["inference_result"] = outputs
    dt = time.perf_counter() - t0
    return {"rows_per_s": len(rows) / dt, "ms_total": 1e3 * dt, "payload_bytes": len(body),
            "rows": len(rows), "cores": 1,
            "what": "handle_data_helper + payload json + write-back (restated reference plumbing)"}


def run_reference_arm(args):
    """`--impl reference`: there is no reference CPU code for this path (the reference
    POSTs to a hosted service), so this arm times the CPU oracle on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from sutro_b200 import modelspec as MS
    from sutro_b200 import vocab as VB
    spec = MS.get_spec(args.model)
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    t0 = time.perf_counter()
    if torch.cuda.is_available():   # drawing 4e9 normals on the host takes minutes; the GPU
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))   # is only a RNG here
        ew = MS.make_engine_weights_on_device(spec, seed=0, device="cuda")
        w = MS.unpack_to_hf(spec, ew)
        del ew
        torch.cuda.empty_cache()
    else:
        w = MS.make_weights(spec, seed=0)
    vocab = VB.build_vocab(spec.family, spec.vocab_size, seed=0)
    setup = time.perf_counter() - t0
    log(f"reference arm: weights + vocab ready in {setup:.1f}s")
    n_sample = args.cpu_rows
    vals = []
    for step in range(args.warmup + args.steps):
        rows = make_rows(n_sample, seed=1000 + step)
        r, _, _ = cpu_baseline(spec, w, vocab, rows, threads, args.cpu_budget_s)
        if step >= args.warmup:
            vals.append(r)
    v = sum(x["value"] for x in vals) / len(vals)
    threads = vals[-1]["cores"]
    line = {"impl": "reference", "metric": "rows_per_sec", "value": v, "unit": "rows/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 * n_sample / v, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": workload_config(args),
            "cpu_baseline": {"value": v, "unit": "rows/s", "cores": threads, "kind": "port",
                             "sample": f"{n_sample} rows per step x {args.steps} steps of the same "
                                       "workload (a bounded sample of the 20k-row frame), CPU oracle "
                                       "(oracle/model_ref.py); the reference repo has no local "
                                       "implementation of this path"},
            "e2e": {"value": v, "unit": "rows/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
            "setup_s": setup}
    emit(line)


def workload_config(args, shape=None):
    wl = ("BASELINE.json configs[1]: one synthetic product-reviews frame per step on rank 0, "
          f"{args.model} bf16, system prompt + Sentiment enum output_schema, greedy, "
          f"max_new_tokens {MAX_NEW}") if WORKLOAD == "sentiment" else (
          f"BASELINE.json configs[2] shape: synthetic documents, {args.model} bf16, "
          "~512-token prompts, exactly 64 generated tokens, no schema, greedy")
    cfg = {"workload": wl, "rows_per_step": args.rows, "model": args.model,
           "weights": "seeded random init (no checkpoints offline)",
           "vocab": "seeded synthetic byte-level BPE",
           "parallelism": f"one replica per GPU x{args.gpus}; the frame's rows are dealt to the "
                          "ranks by byte length (snake order), results gathered in row order on "
                          "rank 0",
           "l2": "inputs_exceed_l2 (8 GB of weights + KV streamed per step; L2 is 126 MB)",
           "max_slots": args.max_slots, "max_prefill_tokens": args.max_prefill_tokens,
           "decoding": "greedy + schema mask, jump-forward (forced JSON syntax is fed with the "
                       "prompt / appended, not decoded token by token)"}
    if shape:
        cfg["shape"] = shape
    return cfg


def frame_shape(eng, rows, stats):
    """Token-level shape of the step's frame, so that rows/s is comparable across rounds."""
    import numpy as np
    from sutro_b200.engine import rows_to_blob
    d_tok, d_toff = eng.tokenizer.encode_blob_dev(*rows_to_blob(rows))
    n = np.diff(d_toff.cpu().numpy())
    pre = stats.get("prefix_cached_tokens", 0)
    forced = stats.get("forced_prefix_tokens", 0)
    n_rows = max(1, len(rows))
    return {"row_text_tokens": {"mean": float(n.mean()), "p5": float(np.percentile(n, 5)),
                                "p50": float(np.percentile(n, 50)),
                                "p95": float(np.percentile(n, 95)), "max": int(n.max())},
            "prompt_tokens_per_row_mean": stats.get("input_tokens", 0) / n_rows,
            "shared_prefix_tokens": int(pre),
            "forced_output_prefix_tokens": int(forced),
            "output_tokens_per_row_mean": stats.get("output_tokens", 0) / n_rows,
            "model_decided_tokens_per_row_mean":
                (stats.get("decode_tokens", 0) + n_rows) / n_rows}


def kernel_block(prof, pk, shared_prefix_tokens=0):
    """Per-class device time of one profiled engine job + the two roofline figures.  Decode
    attention is quoted on NON-SHARED KV bytes only: the shared prefix's pages are read by
    every row and live in L2, so they are not HBM traffic."""
    kms = prof["kernel_ms"]
    tot_ms = sum(kms.values()) or 1.0
    gemm_tf = prof["gemm_flops"] / (kms["gemm"] * 1e-3) / 1e12 if kms["gemm"] else 0.0
    dec_bytes = prof["attn_decode_bytes"]
    shared = float(shared_prefix_tokens) * prof.get("decode_tokens", 0) * \
        prof.get("_kv_bytes_per_token", 0)
    own = max(0.0, dec_bytes - shared)
    gbs = own / (kms["attn_decode"] * 1e-3) / 1e9 if kms["attn_decode"] else 0.0
    return {"kernel_ms": kms, "share": {k: v / tot_ms for k, v in kms.items()},
            "gemm_tflops": gemm_tf, "gemm_frac_of_sustained_peak": gemm_tf / pk["bf16_tflops_sustained"],
            "attn_decode_gbs_non_shared_kv": gbs, "attn_decode_frac_of_hbm_peak": gbs / pk["hbm_gbs"],
            "attn_decode_share_of_step": kms["attn_decode"] / tot_ms}


# ----------------------------------------------------------------------------- secondary configs
def secondary_blocks(args, pk, dev, headline_eng, weights, vocab):
    """configs[2], [3], [4] on one GPU, bounded samples, after the headline's timed region."""
    import torch
    from sutro_b200 import modelspec as MS
    from sutro_b200 import synth
    from sutro_b200 import vocab as VB
    from sutro_b200.engine import LocalEngine
    from sutro_b200.schema_fsm import FsmLimits
    out = {}

    def timed(eng, rows, **kw):
        torch.cuda.synchronize()
        t = time.perf_counter()
        r = eng.infer_one_call(rows, return_tokens=False, **kw)
        return r, time.perf_counter() - t

    # ---- configs[2]: documents, decode-heavy, the headline engine ----
    try:
        kw = dict(system_prompt=None, json_schema=None, max_new_tokens=64, ignore_eos=True)
        spec = headline_eng.spec
        rows = synth.documents(args.docs_rows, seed=11, words=475)
        timed(headline_eng, rows[:256], **kw)
        r, dt = timed(headline_eng, rows, **kw)
        prof = headline_eng.generate(rows[:max(256, args.docs_rows // 2)], profile=True,
                                     return_text=False, **kw).stats
        prof["_kv_bytes_per_token"] = spec.kv_bytes_per_token
        blk = kernel_block(prof, pk, 0)
        blk.update(config="BASELINE.json configs[2] shape: synthetic documents, ~512-token prompts, "
                          "64 generated tokens (ignore_eos), no schema, qwen-3-4b bf16, 1 GPU",
                   rows=len(rows), rows_per_sec=len(rows) / dt,
                   rows_per_sec_device=len(rows) / (r.stats["t_device_ms"] * 1e-3),
                   output_tokens_per_sec=r.stats["output_tokens"] / dt,
                   input_tokens_per_sec=r.stats["input_tokens"] / dt,
                   prompt_tokens_per_row_mean=r.stats["input_tokens"] / len(rows),
                   decode_steps=r.stats["decode_steps"], prefill_steps=r.stats["prefill_steps"],
                   speed_of_light_rows_per_sec=267.0)
        out["configs2_docs"] = blk
        log(f"secondary configs[2]: {blk['rows_per_sec']:.1f} rows/s, decode attention "
            f"{blk['attn_decode_gbs_non_shared_kv']:.0f} GB/s at {100 * blk['attn_decode_share_of_step']:.1f}% of the step")
    except Exception as e:  # a secondary block must not sink the headline
        out["configs2_docs"] = {"failed": repr(e)}
    headline_eng.close()
    del headline_eng, weights
    torch.cuda.empty_cache()

    # ---- configs[3]: embeddings, prefill only ----
    try:
        spec = MS.get_spec("qwen-3-embedding-0.6b")
        w = MS.make_engine_weights_on_device(spec, seed=0, device=dev)
        v = VB.build_vocab(spec.family, spec.vocab_size, seed=0)
        eng = LocalEngine(spec, w, v, device=dev, max_slots=4096, max_prefill_tokens=32768,
                          kv_pages=32768)
        rows = synth.short_texts(args.embed_rows, seed=2)
        timed(eng, rows[:20000])
        r, dt = timed(eng, rows)
        prof = eng.generate(rows[:50000], profile=True).stats
        kms = prof["kernel_ms"]
        gemm_tf = prof["gemm_flops"] / (kms["gemm"] * 1e-3) / 1e12 if kms["gemm"] else 0.0
        out["configs3_embed"] = {
            "config": "BASELINE.json configs[3] shape: short texts (8-64 tokens), "
                      "qwen-3-embedding-0.6b, prefill only, last-token pool + L2 normalise, fp32 "
                      "[N,1024] out, 1 GPU",
            "rows": len(rows), "rows_per_sec": len(rows) / dt,
            "rows_per_sec_device": len(rows) / (r.stats["t_device_ms"] * 1e-3),
            "input_tokens_per_sec": r.stats["input_tokens"] / dt,
            "prompt_tokens_per_row_mean": r.stats["input_tokens"] / len(rows),
            "phase_ms": {k: r.stats[k] for k in ("t_h2d_ms", "t_device_ms", "t_d2h_ms")},
            "host_s_outside_the_c_call": r.stats["t_total_s"] - r.stats["t_call_s"],
            "d2h_bytes": r.stats["d2h_bytes"], "kernel_ms": kms, "gemm_tflops": gemm_tf,
            "gemm_frac_of_sustained_peak": gemm_tf / pk["bf16_tflops_sustained"],
            "embedding_norm_check": float((r.embeddings[:64] ** 2).sum(1).mean())}
        log(f"secondary configs[3]: {out['configs3_embed']['rows_per_sec']:.0f} rows/s")
        eng.close()
        del eng, w
        torch.cuda.empty_cache()
    except Exception as e:
        out["configs3_embed"] = {"failed": repr(e)}

    # ---- configs[4]: llama-3.1-8b, nested schema ----
    try:
        spec = MS.get_spec("llama-3.1-8b")
        w = MS.make_engine_weights_on_device(spec, seed=0, device=dev)
        v = VB.build_vocab(spec.family, spec.vocab_size, seed=0)
        eng = LocalEngine(spec, w, v, device=dev, max_slots=2048, max_prefill_tokens=32768)
        lim = FsmLimits(max_string_chars=12, max_array_items=3)
        kw = dict(system_prompt="Extract the order as JSON.", json_schema=ORDER_SCHEMA,
                  max_new_tokens=128, fsm_limits=lim)
        rows = synth.extraction_documents(args.extract_rows, seed=3)
        timed(eng, rows[:128], **kw)
        r, dt = timed(eng, rows, **kw)
        valid = 0
        for o in r.outputs:
            try:
                d = json.loads(o)
                valid += int(isinstance(d, dict) and set(d) >= {"customer", "items", "paid"})
            except ValueError:
                pass
        prof = eng.generate(rows[:max(128, args.extract_rows // 2)], profile=True,
                            return_text=False, **kw).stats
        prof["_kv_bytes_per_token"] = spec.kv_bytes_per_token
        blk = kernel_block(prof, pk, prof.get("prefix_cached_tokens", 0))
        blk.update(config="BASELINE.json configs[4] shape: pseudo-documents (~300 prompt tokens), "
                          "llama-3.1-8b bf16, nested output_schema (object -> list of objects -> "
                          "{str, int(min,max), enum, optional float}), greedy + FSM mask with "
                          "jump-forward, cap 128 tokens, 1 GPU",
                   rows=len(rows), rows_per_sec=len(rows) / dt,
                   rows_per_sec_device=len(rows) / (r.stats["t_device_ms"] * 1e-3),
                   output_tokens_per_sec=r.stats["output_tokens"] / dt,
                   model_decided_tokens_per_sec=(r.stats["decode_tokens"] + len(rows)) / dt,
                   input_tokens_per_sec=r.stats["input_tokens"] / dt,
                   prompt_tokens_per_row_mean=r.stats["input_tokens"] / len(rows),
                   outputs_valid_json_objects=f"{valid}/{len(rows)}",
                   fsm_states=r.stats["fsm_states"], decode_steps=r.stats["decode_steps"])
        out["configs4_extraction"] = blk
        log(f"secondary configs[4]: {blk['rows_per_sec']:.1f} rows/s, {valid}/{len(rows)} valid")
        eng.close()
        del eng, w
        torch.cuda.empty_cache()
    except Exception as e:
        out["configs4_extraction"] = {"failed": repr(e)}
    return out


# ----------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="qwen-3-4b")
    ap.add_argument("--rows", type=int, default=20000, help="rows of the frame (whole job) per step")
    ap.add_argument("--workload", default="sentiment", choices=["sentiment", "docs"],
                    help="sentiment = BASELINE.json configs[1] (the headline); docs = configs[2] "
                         "shape (~512-token prompts, 64 generated tokens, no schema)")
    ap.add_argument("--max-slots", type=int, default=3584,
                    help="decode slots; 3584 = 14 x 256 rows quantises the CTA-pair GEMM tiles well")
    ap.add_argument("--max-prefill-tokens", type=int, default=32768)
    ap.add_argument("--cpu-rows", type=int, default=8, help="max rows in the CPU-baseline sample")
    ap.add_argument("--cpu-budget-s", type=float, default=25.0,
                    help="stop the CPU-baseline sample after this many seconds of CPU work")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true",
                    help="skip the configs[2]/[3]/[4] secondary blocks")
    ap.add_argument("--docs-rows", type=int, default=2048)
    ap.add_argument("--embed-rows", type=int, default=200000)
    ap.add_argument("--extract-rows", type=int, default=1024)
    ap.add_argument("--kv-pages", type=int, default=None,
                    help="KV pool size in pages (default: 80%% of free memory); small pools keep "
                         "ncu's save/restore cheap")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's result column to DIR as "
                         ".npy (code points as float32, at most 64 MB; a seeded row sample if "
                         "larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU arm computed (--impl ours)")
    global WORKLOAD
    WORKLOAD = args.workload
    divert_stdout()
    if args.impl == "reference":
        return run_reference_arm(args)

    import pandas as pd
    import torch
    import torch.distributed as dist
    from sutro_b200 import modelspec as MS
    from sutro_b200 import vocab as VB
    from sutro_b200.engine import LocalEngine
    from sutro_b200.sdk import Sutro

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    spec = MS.get_spec(args.model)
    pk = peaks()

    # ---- weights: rank 0 draws them, everyone else receives them over NCCL/NVLink ----
    t0 = time.perf_counter()
    weights = MS.make_engine_weights_on_device(spec, seed=0 if rank == 0 else 1 + rank, device=dev)
    bcast_ms = None
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        tb = time.perf_counter()
        for t in weights.all_tensors():
            dist.broadcast(t, src=0)
        torch.cuda.synchronize()
        bcast_ms = (time.perf_counter() - tb) * 1e3
    vocab = VB.build_vocab(spec.family, spec.vocab_size, seed=0)
    eng = LocalEngine(spec, weights, vocab, device=dev, max_slots=args.max_slots,
                      max_prefill_tokens=args.max_prefill_tokens, kv_pages=args.kv_pages)
    # results cache private to this run: a fixed path under /tmp may belong to another user
    cache = tempfile.TemporaryDirectory(prefix="sb200-bench-cache-")
    client = Sutro(verbose=False, cache_dir=cache.name)
    client.register_engine(args.model, eng)
    setup_s = time.perf_counter() - t0
    log(f"engine ready in {setup_s:.1f}s (kv_pages={eng.kv_pages})")

    def fence():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the frames exist before infer() is called: row generation (pure Python) is hoisted out
    # of the timed region; only rank 0 holds them
    n_frames = args.warmup + args.steps
    frames = [pd.DataFrame({COLUMN: make_rows(args.rows, seed=7919 + i)}) if rank == 0 else None
              for i in range(n_frames)]
    log(f"{n_frames} frames of {args.rows} rows generated")
    kw = infer_kwargs(args.model)

    def step(i):
        """the user's call; returns the job's stats on rank 0"""
        data = frames[i] if rank == 0 else []
        job_id = client.infer(data, **kw)
        if job_id is None:
            raise RuntimeError("infer() failed: " + str(
                [j.failure_reason for j in client._jobs.values()][-1:]))
        return client._jobs[job_id].stats

    for i in range(args.warmup):
        t = time.perf_counter()
        st = step(i)
        if rank == 0:
            log(f"warmup {i}: {time.perf_counter() - t:.2f}s (prefill_steps "
                f"{st.get('prefill_steps')}, decode_steps {st.get('decode_steps')})")
    clocks = ClockSampler(local)
    fence()
    clocks.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    t_start = time.perf_counter()
    stats = []
    for i in range(args.steps):
        t = time.perf_counter()
        stats.append(step(args.warmup + i))
        log(f"step {i}: {time.perf_counter() - t:.2f}s")
    ev1.record()
    fence()
    t_e2e = time.perf_counter() - t_start
    clk = clocks.stop()

    # ---- counters: rank 0 holds the job-wide numbers (sharded stats are already aggregated) ----
    tt = torch.tensor([t_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_e2e_max = float(tt[0])
    line = None
    if rank == 0:
        t_dev = sum(s["t_device_ms"] for s in stats) * 1e-3
        n_out = sum(s["output_tokens"] for s in stats)
        n_in = sum(s["input_tokens"] for s in stats)
        n_dec = sum(s["decode_tokens"] + args.rows for s in stats)

        def launches_of(s):
            per = s.get("per_gpu") or [s]
            return sum(sum(p["kernel_launches"].values()) + p.get("tokenizer_launches", 0)
                       for p in per if p) + (3 * 2 if s.get("per_gpu") else 0)  # + row selection
        launches = sum(launches_of(s) for s in stats)
        total_rows = args.rows * args.steps
        outputs = list(frames[-1]["inference_result"])
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs,
                         dump_width(vocab, gen_kwargs()["max_new_tokens"]))
        if WORKLOAD == "sentiment":
            ok = all(json.loads(o)["sentiment"] in ("positive", "neutral", "negative")
                     for i in range(args.warmup, n_frames)
                     for o in frames[i]["inference_result"][:512])
        else:
            ok = all(s["output_tokens"] == 64 * args.rows for s in stats)

    # ---- one extra profiled job on rank 0 (a shard-sized sample at N > 1): per-kernel-class
    #      device time (CUDA events on the engine stream) for the roofline numbers ----
    if rank == 0:
        log("timed region done; profiled job")
        sample = list(frames[-1][COLUMN])[:max(1, args.rows // world)]
        prof = eng.generate(sample, profile=True, **gen_kwargs()).stats
        prof["_kv_bytes_per_token"] = spec.kv_bytes_per_token
        kb = kernel_block(prof, pk, prof.get("prefix_cached_tokens", 0))
        kms = prof["kernel_ms"]
        roofline = {"kernel": "gemm_bf16_tn_kernel / gemm2_bf16_tn_kernel (tcgen05)",
                    "bound": "tensor", "achieved": kb["gemm_tflops"],
                    "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                    "frac": kb["gemm_frac_of_sustained_peak"],
                    "traffic": ncu_traffic("r02_ncu_prefill_step.csv", "gemm2_bf16_tn_kernel<2, 7"),
                    "traffic_note": "bytes of ONE gate/up GEMM launch of a full prefill step "
                                    "(M=32670, N=19456, K=2560; algorithmic 903 MB = A 167 + "
                                    "W 100 + SwiGLU output 636; W does not fit L2, so A and W "
                                    "are re-read) from the committed capture "
                                    "profiles/r02_ncu_prefill_step.csv, not from this run",
                    "peak_source": pk["source"] + " (sustained: kernel timed inside a long step)",
                    "share_of_step": kb["share"]["gemm"],
                    "launches": prof["kernel_launches"]["gemm"],
                    "avg_launch_ms": kms["gemm"] / max(1, prof["kernel_launches"]["gemm"]),
                    "algorithmic_flops": prof["gemm_flops"]}
        roofline_attn = {"kernel": "attn_decode_warp_kernel", "bound": "hbm",
                         "achieved": kb["attn_decode_gbs_non_shared_kv"], "peak": pk["hbm_gbs"],
                         "unit": "GB/s", "frac": kb["attn_decode_frac_of_hbm_peak"],
                         "bytes": "non-shared KV only (the shared system-prompt pages are L2 hits)",
                         "traffic": ncu_traffic("r02_ncu_decode_side.csv", "attn_decode_warp_kernel"),
                         "share_of_step": kb["attn_decode_share_of_step"],
                         "launches": prof["kernel_launches"]["attn_decode"],
                         "note": "the headline job barely decodes (jump-forward); the graded "
                                 "decode-attention number is secondary.configs2_docs"}
        shape = frame_shape(eng, list(frames[-1][COLUMN]), stats[-1] if world == 1 else
                            {**stats[-1], **{k: prof[k] for k in ("prefix_cached_tokens",
                                                                    "forced_prefix_tokens")}})

        cpu = None
        if world == 1 and not args.no_cpu_baseline and WORKLOAD == "sentiment":
            try:
                log("cpu baseline: copying weights to host")
                hf_w = MS.unpack_to_hf(spec, weights)
                log("cpu baseline: running oracle")
                rows8 = list(frames[-1][COLUMN])[:args.cpu_rows]
                cpu, texts, margins = cpu_baseline(spec, hf_w, vocab, rows8, os.cpu_count() or 1,
                                                   args.cpu_budget_s)
                del hf_w
                # the checker's verdict travels with the number: the same rows through the engine
                got = outputs[:len(texts)]
                eq = [a == b for a, b in zip(got, texts)]
                cpu["outputs_equal"] = f"{sum(eq)}/{len(eq)}"
                cpu["mismatch_min_margins"] = [m for m, e in zip(margins, eq) if not e]
                # a row whose oracle run passed through a decision closer than the near-tie
                # band of the parity tests (0.06 logit units, tests/test_engine_gpu.py) may
                # legitimately come out differently: both arms round a 36-layer bf16 network
                near = sum(1 for m, e in zip(margins, eq) if not e and m is not None and m < 0.06)
                cpu["near_tie_band"] = 0.06
                cpu["outputs_equal_or_inside_near_tie_band"] = f"{sum(eq) + near}/{len(eq)}"
                cpu["engine_outputs_sample"] = got[:3]
                log(f"cpu baseline done: {cpu['value']:.3f} rows/s, outputs equal {cpu['outputs_equal']}")
            except Exception as e:  # the baseline must not sink the benchmark line
                cpu = {"value": None, "unit": "rows/s", "cores": os.cpu_count(), "kind": "port",
                       "sample": f"failed: {e!r}"}
        try:
            plumbing = plumbing_cost(args.model, list(frames[-1][COLUMN]), outputs)
        except Exception as e:
            plumbing = {"failed": repr(e)}
        st = stats[-1]
        line = {
            "metric": "rows_per_sec", "value": total_rows / t_dev, "unit": "rows/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * t_dev / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": workload_config(args, shape),
            "timing": {"value": "CUDA events: column resident in rank 0's HBM -> ordered results "
                                "resident in rank 0's HBM (N>1: incl. NCCL broadcast, slowest rank, "
                                "NCCL gather, ordered merge)",
                       "e2e": "wall clock of the K public-API calls between barrier+synchronize, "
                              "max over ranks; host frame in, result column written back"},
            "output_tokens_per_sec": n_out / t_dev,
            "model_decided_tokens_per_sec": n_dec / t_dev,
            "input_tokens_per_sec": n_in / t_dev,
            "e2e": {"value": total_rows / t_e2e_max, "unit": "rows/s",
                    "h2d_bytes_per_step": st["h2d_bytes"], "d2h_bytes_per_step": st["d2h_bytes"],
                    "ms_per_step": 1e3 * t_e2e_max / args.steps,
                    "cuda_event_ms_total": ev0.elapsed_time(ev1),
                    "api": "sutro_b200.sdk.Sutro.infer(df, column=, model=, system_prompt=, "
                           "output_schema=) -> " + ("sb200_infer_text (one C-ABI call)" if world == 1
                                                    else "sharding.infer_frame_sharded over NCCL")},
            "gpu_launches": int(launches),
            "roofline": roofline, "roofline_attn_decode": roofline_attn,
            "kernel_ms_profiled_job": kms,
            "cpu_baseline": cpu, "host_plumbing": plumbing, "clocks": clk,
            "outputs_valid": bool(ok),
            "job": {k: st.get(k) for k in ("prefill_steps", "decode_steps", "input_tokens",
                                           "output_tokens", "decode_tokens", "n_gpus")},
            "setup_s": setup_s, "weight_broadcast_ms": bcast_ms, "kv_pages": eng.kv_pages,
        }
        if world == 1:
            line["phase_ms_last_step"] = {k: st[k] for k in ("t_h2d_ms", "t_device_ms", "t_d2h_ms")}
        else:
            line["sharding"] = {
                "rows_per_rank": [p["n_rows"] if p else 0 for p in st["per_gpu"]],
                "engine_s_per_rank_last_step": [round(p["t_engine_s"], 4) if p else 0.0
                                                for p in st["per_gpu"]],
                "limiting_term": "max over ranks of the shard's engine time (tail imbalance) vs "
                                 "broadcast+gather: see engine_s_per_rank_last_step against ms_per_step"}
    if world == 1 and not args.no_secondary and WORKLOAD == "sentiment":
        line["secondary"] = secondary_blocks(args, pk, dev, eng, weights, vocab)
    if rank == 0:
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
