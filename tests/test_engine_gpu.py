"""End-to-end parity of the engine (through the C-ABI) against the CPU oracle on tiny
architectures: tokenizer ids bit-exact, greedy token ids equal wherever the oracle's
top-1 margin is not a near-tie, constrained outputs valid and equal, embeddings close.

Tolerances (stated once, used below):
  MARGIN_EPS   a greedy decision must equal the oracle's whenever the oracle's top-1/top-2
               logit gap exceeds 0.06 (logit std is ~1; two bf16 pipelines that differ only
               in fp32 summation order disagree by ~0.02 on these tiny models).  Below that
               gap the engine may pick another token whose oracle logit is within 0.06 of the
               oracle's best (a near-tie flip); anything else fails.  After a flip the
               sequences legitimately diverge, so the comparison stops there.  Every flip is
               recorded (FLIP_LOG) and the counts are printed and bounded per test.
  EMB_TOL      embedding vectors: max abs diff 2e-2 on unit-norm vectors.
"""
import json
from typing import List, Literal

import numpy as np
import pytest
import torch
from pydantic import BaseModel, Field

from oracle.bpe_ref import RefTokenizer
from oracle.fsm_ref import TokenFSM
from oracle.model_ref import RefModel
from sutro_b200 import modelspec as MS
from sutro_b200 import synth, vocab as VB
from sutro_b200.schema_fsm import FsmLimits, compile_schema

pytestmark = pytest.mark.gpu

MARGIN_EPS = 0.06
EMB_TOL = 2e-2
SYS = synth.README_SYSTEM_PROMPT


class SentimentEnum(BaseModel):
    sentiment: Literal["positive", "neutral", "negative"]


class Extract(BaseModel):
    name: str = Field(max_length=8)
    qty: int = Field(ge=0, le=20)
    tags: List[Literal["a", "b"]] = Field(max_length=2)


def build(name, seed=0, **kw):
    from sutro_b200.engine import LocalEngine
    spec = MS.get_spec(name)
    w = MS.make_weights(spec, seed=seed, std=0.05)
    v = VB.build_vocab(spec.family, spec.vocab_size, seed=0, n_trained=600)
    eng = LocalEngine(spec, MS.pack_for_engine(spec, w, "cuda"), v, device=0, kv_pages=512, **kw)
    return spec, w, v, eng


def compare_greedy(got: List[int], ref, label="", eos_id=-1):
    """Returns (#decisions verified equal, #decisions the oracle made, #near-tie flips).
    Tokens the automaton forces (jump-forward prefix / tails) are not decisions and must
    match exactly; a decision may differ only as a near-tie flip to the oracle's runner-up."""
    toks = list(ref.tokens) + ([eos_id] if ref.finished_by == "eos" else [])
    dec = {pos: i for i, pos in enumerate(ref.decision_pos)}
    for i, want in enumerate(toks):
        have = got[i] if i < len(got) else eos_id          # the engine stopped: it chose EOS
        if have == want:
            continue
        assert i in dec, (label, "forced token differs", i, got, ref.tokens)
        d = dec[i]
        assert ref.margins[d] < MARGIN_EPS, (label, i, got, ref.tokens, ref.margins)
        # the engine's pick must itself be within the near-tie band of the oracle's best
        # (several candidates can sit inside it at once)
        gap = ref.near[d].get(have)
        assert gap is not None and gap < MARGIN_EPS, (label, i, have, ref.near[d])
        FLIP_LOG.append((label, round(ref.margins[d], 4), round(gap, 4)))
        return d, len(ref.margins), 1
    return len(ref.margins), len(ref.margins), 0


FLIP_LOG = []     # (row, oracle top-1 margin, oracle gap of the engine's pick) of every near-tie flip


def record_parity(test: str, rows: int, compared: int, total: int, flips: int):
    """One line per parity test run: how many greedy decisions were checked against the oracle
    and how many near-tie flips were seen (appended to gpurun_out/parity_flips.jsonl so that
    the numbers behind the tolerance travel back from the GPU box; also printed)."""
    import os
    rec = {"test": test, "rows": rows, "decisions_verified": compared, "decisions_total": total,
           "near_tie_flips": flips, "margin_eps": MARGIN_EPS,
           "flips": [list(f) for f in FLIP_LOG[-flips:]] if flips else []}
    print("PARITY", json.dumps(rec))
    out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    try:
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, "parity_flips.jsonl"), "a") as f:
            f.write(json.dumps(rec) + "\n")
    except OSError:
        pass


# rows (of 15) allowed to hit a near-tie flip within their first 12 decisions; measured counts
# are in profiles/r02_parity_flips.jsonl (seeded tiny random models have flat logits: a 12-token
# greedy run crosses a < 0.06 margin in roughly one row out of three)
MAX_FLIP_ROWS = 7

ROWS = synth.README_REVIEWS + synth.product_reviews(9, seed=7) + ["", "x", "ok ok ok"]


@pytest.mark.parametrize("name", ["tiny-qwen3", "tiny-llama"])
def test_gpu_tokenizer_matches_oracle(name):
    spec, w, v, eng = build(name)
    ref = RefTokenizer(v)
    texts = ROWS + synth.extraction_documents(5, seed=2) + [
        "unicode: café naïve Straße 東京 Привет мир ١٢٣ ½ 🙂 end", "tabs\tand\nnewlines\r\n\r\n  x ",
        "don't DON'T we'LL they've I'm", "numbers 1234567 3.14 v2.1", "x" * 200, "   ", "\n\n a"]
    got = eng.tokenizer.encode(texts)
    for t, g in zip(texts, got):
        assert g == ref.encode(t), repr(t)
    tpl = VB.chat_template(spec.family, SYS)
    assert eng.tokenizer.encode_pieces(tpl.prefix) == ref.encode_pieces(tpl.prefix)
    # detokenizer round trip
    d_tok, d_off = eng.tokenizer.encode_blob_dev(*__import__("sutro_b200.engine", fromlist=["x"])
                                                 .rows_to_blob(texts))
    n = int(d_off[-1].item())
    b, boff = eng.tokenizer.decode_dev(d_tok[:n].contiguous(), d_off)
    for i, t in enumerate(texts):
        assert b[boff[i]:boff[i + 1]].tobytes() == t.encode("utf-8")


def test_gpu_tokenizer_honours_ignore_merges(tmp_path):
    """A tokenizer file with model.ignore_merges (Llama-3): pre-tokens that are vocabulary
    entries come out as that entry — the GPU tokenizer (whole-word override table) against the
    oracle and against `tokenizers` reading the same file."""
    from test_pretrained_cpu import ROWS_TXT, ignore_merges_vocab, override_texts
    from sutro_b200.engine import GpuTokenizer
    _, hf, loaded = ignore_merges_vocab(tmp_path)
    tok = GpuTokenizer(loaded, torch.device("cuda:0"))
    ref = RefTokenizer(loaded)
    texts = override_texts(loaded) + ROWS_TXT + ROWS
    hits = 0
    for t, g in zip(texts, tok.encode(texts)):
        assert g == ref.encode(t), repr(t)
        assert loaded.to_real_ids(g) == hf.encode(t, add_special_tokens=False).ids, repr(t)
        hits += len(g) == 1 and any(g[0] == e for _, e in loaded.word_overrides)
    assert hits >= 3
    # the same vocabulary without the flag: the table is empty and plain BPE comes back
    import dataclasses
    plain_v = dataclasses.replace(loaded, word_overrides=None)
    plain = GpuTokenizer(plain_v, torch.device("cuda:0"))
    ref_plain = RefTokenizer(plain_v)
    for t, g in zip(texts, plain.encode(texts)):
        assert g == ref_plain.encode(t), repr(t)


@pytest.mark.parametrize("name", ["tiny-qwen3", "tiny-qwen3-g4", "tiny-llama"])
def test_unconstrained_greedy_matches_oracle(name):
    spec, w, v, eng = build(name, max_slots=8, max_prefill_tokens=512)
    res = eng.generate(ROWS, system_prompt=SYS, max_new_tokens=12, ignore_eos=True,
                       return_tokens=True)
    ref_tok, model = RefTokenizer(v), RefModel(spec, w)
    tpl = VB.chat_template(spec.family, SYS)
    compared = total = flips = 0
    for row, got in zip(ROWS, res.out_tokens):
        prompt = ref_tok.render(tpl, row, spec.max_position - 12)
        r = model.generate(prompt, 12, v.eos_id, ignore_eos=True)
        assert len(got) == 12
        c, t, f = compare_greedy(got, r, row[:30], v.eos_id)
        compared, total, flips = compared + c, total + t, flips + f
    record_parity(f"unconstrained_greedy[{name}]", len(ROWS), compared, total, flips)
    assert compared >= 0.5 * total, (compared, total)   # the criterion is not vacuous
    assert flips <= MAX_FLIP_ROWS, flips
    assert res.stats["rows_done"] == len(ROWS)
    assert res.stats["prefix_cached_tokens"] >= 16       # the system prompt was shared


LOGIT_RMS_TOL = 0.03     # x logit std: rms(engine - oracle) over the vocabulary
LOGIT_MAX_TOL = 0.15     # x logit std: worst single logit


@pytest.mark.parametrize("name", ["tiny-qwen3", "tiny-qwen3-g4", "tiny-llama"])
def test_teacher_forced_logits_within_tolerance(name):
    """First-decision logits (fp32) of every row against the oracle's, same prompt."""
    spec, w, v, eng = build(name, max_slots=8, max_prefill_tokens=512)
    res = eng.generate(ROWS, system_prompt=SYS, max_new_tokens=1, ignore_eos=True,
                       return_tokens=True, return_first_logits=True)
    ref_tok, model = RefTokenizer(v), RefModel(spec, w)
    tpl = VB.chat_template(spec.family, SYS)
    worst_rms = worst_max = 0.0
    for i, row in enumerate(ROWS):
        want = model.logits(ref_tok.render(tpl, row, spec.max_position - 1))[-1]
        got = res.first_logits[i]
        std = want.std().item()
        d = (got - want).abs()
        worst_rms = max(worst_rms, d.pow(2).mean().sqrt().item() / std)
        worst_max = max(worst_max, d.max().item() / std)
    assert worst_rms < LOGIT_RMS_TOL and worst_max < LOGIT_MAX_TOL, (worst_rms, worst_max)


def test_prefix_sharing_and_batch_geometry_do_not_change_results():
    spec, w, v, eng = build("tiny-qwen3-g4", max_slots=32, max_prefill_tokens=1024)
    rows = synth.product_reviews(40, seed=11)
    a = eng.generate(rows, system_prompt=SYS, max_new_tokens=6, ignore_eos=True,
                     return_tokens=True).out_tokens
    b = eng.generate(rows, system_prompt=SYS, max_new_tokens=6, ignore_eos=True,
                     return_tokens=True, share_prefix=False).out_tokens
    eng.close()
    spec, w, v, eng2 = build("tiny-qwen3-g4", max_slots=4, max_prefill_tokens=300,
                             min_admit_rows=1)
    c = eng2.generate(rows, system_prompt=SYS, max_new_tokens=6, ignore_eos=True,
                      return_tokens=True).out_tokens
    same_ab = sum(x == y for x, y in zip(a, b))
    same_ac = sum(x == y for x, y in zip(a, c))
    record_parity("batch_geometry(share_prefix off / 4 slots)", len(rows), same_ab, same_ac, 0)
    # a different batch geometry (slots, prefill packing, admission order) must not change a
    # single token: no kernel choice depends on the batch.  Without prefix sharing the prefix
    # is recomputed inside each row's own KV blocks — another summation order, so near-tie
    # decisions may move.
    assert same_ac == 40, same_ac
    assert same_ab >= 36, same_ab


@pytest.mark.parametrize("jump", [True, False])
@pytest.mark.parametrize("schema_model", [SentimentEnum, Extract])
def test_schema_constrained_outputs_validate_and_match_oracle(schema_model, jump):
    """jump=True: forced output prefix rides with the prompt and forced terminal tails are
    appended without a forward pass (engine default); jump=False: plain masked greedy."""
    spec, w, v, eng = build("tiny-qwen3", max_slots=8, max_prefill_tokens=512)
    schema = schema_model.model_json_schema()
    lim = FsmLimits(max_string_chars=8, max_array_items=2)
    res = eng.generate(ROWS, system_prompt=SYS, json_schema=schema, max_new_tokens=64,
                       fsm_limits=lim, return_tokens=True, jump_forward=jump)
    assert res.stats["jump_forward"] == jump
    dfa = compile_schema(schema, lim)
    fsm = TokenFSM(dfa, v)
    ref_tok, model = RefTokenizer(v), RefModel(spec, w)
    if jump:
        assert fsm.enable_jump_forward(ref_tok)
        assert res.stats["forced_prefix_tokens"] == len(fsm.forced_prefix) > 0
    tpl = VB.chat_template(spec.family, SYS)
    compared = total = flips = 0
    for row, text, got in zip(ROWS, res.outputs, res.out_tokens):
        obj = json.loads(text)                       # every output is valid JSON ...
        schema_model.model_validate(obj)             # ... and an instance of the schema
        assert dfa.matches(text.encode("utf-8"))
        max_prompt = spec.max_position - 64 - len(fsm.forced_prefix)
        r = model.generate(ref_tok.render(tpl, row, max_prompt), 64, v.eos_id, fsm=fsm)
        c, t, f = compare_greedy(got, r, row[:30], v.eos_id)
        compared, total, flips = compared + c, total + t, flips + f
    record_parity(f"schema[{schema_model.__name__},jump={jump}]", len(ROWS), compared, total, flips)
    assert compared >= 0.5 * total, (compared, total)
    assert flips <= MAX_FLIP_ROWS, flips
    if jump:  # fewer forward passes: the sentiment rows need 1-2 decisions each
        assert res.stats["decode_tokens"] < sum(len(t) for t in res.out_tokens)


def test_max_new_tokens_truncates_and_eos_stops():
    spec, w, v, eng = build("tiny-qwen3", max_slots=8, max_prefill_tokens=512)
    res = eng.generate(ROWS[:4], max_new_tokens=3, return_tokens=True)
    assert all(len(t) <= 3 for t in res.out_tokens)
    # a row longer than the context window is truncated (truncate_rows=True) ...
    long_row = "word " * 2000
    res = eng.generate([long_row, "short"], max_new_tokens=4, ignore_eos=True, return_tokens=True)
    assert res.stats["rows_truncated"] == 1 and len(res.out_tokens[0]) == 4
    # ... or rejected (truncate_rows=False)
    from sutro_b200._lib import Sb200Error
    with pytest.raises(Sb200Error, match="truncate_rows=False"):
        eng.generate([long_row], max_new_tokens=4, truncate_rows=False)


@pytest.mark.parametrize("T,k,p", [(1.0, 0, 1.0), (0.7, 20, 1.0), (1.3, 0, 0.8), (0.9, 50, 0.9)])
def test_sampling_matches_oracle_on_the_engine_logits(T, k, p):
    """temperature / top-k / top-p: the sampler is checked against the numpy oracle on the
    engine's own first-decision logits (same Philox draw); a disagreement is tolerated only
    when the draw sits within fp32 rounding of a CDF boundary."""
    from oracle import sampler_ref as SR
    spec, w, v, eng = build("tiny-qwen3", max_slots=16, max_prefill_tokens=1024)
    rows = ROWS * 4
    res = eng.generate(rows, system_prompt=SYS, max_new_tokens=1, ignore_eos=True,
                       return_tokens=True, return_first_logits=True, temperature=T, top_k=k,
                       top_p=p, seed=123, seed_per_row=True, return_logprobs=True)
    allowed = np.ones(spec.vocab_size, dtype=bool)
    allowed[v.n_regular:] = True
    near_boundary = 0
    for i in range(len(rows)):
        lg = res.first_logits[i].numpy()
        u = SR.uniform(123, i, 0, True)
        tok, slack = SR.sample(lg, allowed, T, k, p, u)
        got = res.out_tokens[i][0]
        if got != tok:
            assert slack < 1e-4, (i, got, tok, slack)
            near_boundary += 1
        keep, _ = SR.kept_set(lg, allowed, T, k, p)
        assert keep[got], (i, got)
        assert abs(res.cum_logprobs[i] - SR.logprob(lg, allowed, T, got)) < 2e-3
    assert near_boundary <= 2


def test_sampling_edge_settings_and_seeding():
    spec, w, v, eng = build("tiny-qwen3", max_slots=16, max_prefill_tokens=1024)
    rows = ["same prompt"] * 12
    greedy = eng.generate(rows, max_new_tokens=6, ignore_eos=True, return_tokens=True).out_tokens
    k1 = eng.generate(rows, max_new_tokens=6, ignore_eos=True, return_tokens=True,
                      temperature=1.0, top_k=1, seed=9, seed_per_row=True).out_tokens
    assert k1 == greedy                                   # top_k = 1 is the arg-max
    shared = eng.generate(rows, max_new_tokens=6, ignore_eos=True, return_tokens=True,
                          temperature=1.5, seed=9, seed_per_row=False).out_tokens
    assert all(t == shared[0] for t in shared)            # one stream -> identical rows agree
    per_row = eng.generate(rows, max_new_tokens=6, ignore_eos=True, return_tokens=True,
                           temperature=1.5, seed=9, seed_per_row=True).out_tokens
    assert len({tuple(t) for t in per_row}) > 6           # own stream per row
    again = eng.generate(rows, max_new_tokens=6, ignore_eos=True, return_tokens=True,
                         temperature=1.5, seed=9, seed_per_row=True).out_tokens
    assert again == per_row                               # reproducible
    # sampling under a schema still yields valid instances
    res = eng.generate(ROWS, system_prompt=SYS, json_schema=Extract.model_json_schema(),
                       max_new_tokens=64, temperature=1.2, top_p=0.95, seed=3, seed_per_row=True,
                       fsm_limits=FsmLimits(max_string_chars=8, max_array_items=2))
    for o in res.outputs:
        Extract.model_validate(json.loads(o))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_in_process_multi_gpu_matches_single_gpu():
    """MultiGpuEngine: replicas on cuda:0 and cuda:1, rows sharded, outputs positional."""
    from sutro_b200.engine import LocalEngine, MultiGpuEngine
    spec = MS.get_spec("tiny-qwen3")
    w = MS.make_weights(spec, seed=0, std=0.05)
    v = VB.build_vocab(spec.family, spec.vocab_size, seed=0, n_trained=600)
    e0 = LocalEngine(spec, MS.pack_for_engine(spec, w, "cuda:0"), v, device=0, kv_pages=256,
                     max_slots=8, max_prefill_tokens=512)
    w1 = MultiGpuEngine._replicate(spec, e0.weights, torch.device("cuda", 1))
    e1 = LocalEngine(spec, w1, v, device=1, kv_pages=256, max_slots=8, max_prefill_tokens=512)
    rows = synth.product_reviews(21, seed=4)
    kw = dict(system_prompt=SYS, json_schema=SentimentEnum.model_json_schema(), max_new_tokens=32,
              return_tokens=True)
    single = e0.generate(rows, **kw)
    multi = MultiGpuEngine([e0, e1]).generate(rows, **kw)
    assert multi.stats["n_gpus"] == 2 and multi.stats["n_rows"] == 21
    assert multi.outputs == single.outputs and multi.out_tokens == single.out_tokens
    # sampled decoding with per-row streams: the draws follow the row's index in the whole job
    skw = dict(system_prompt=SYS, max_new_tokens=12, return_tokens=True, temperature=0.9,
               top_k=20, seed=5, seed_per_row=True, return_logprobs=True)
    s1 = e0.generate(rows, **skw)
    for balance in ("bytes", "rows"):
        s2 = MultiGpuEngine([e0, e1]).generate(rows, balance=balance, **skw)
        assert s2.out_tokens == s1.out_tokens
        assert np.allclose(s2.cum_logprobs, s1.cum_logprobs, atol=1e-3)


def test_row_ids_key_the_per_row_random_streams():
    """A shard that passes the rows' job-wide indices draws what the unsharded job draws."""
    spec, w, v, eng = build("tiny-qwen3", max_slots=16, max_prefill_tokens=1024)
    rows = synth.product_reviews(12, seed=9)
    kw = dict(system_prompt=SYS, max_new_tokens=10, return_tokens=True, temperature=1.0,
              seed=3, seed_per_row=True)
    whole = eng.generate(rows, **kw)
    part = eng.generate(rows[5:], row_ids=list(range(5, 12)), **kw)
    assert part.out_tokens == whole.out_tokens[5:]
    local = eng.generate(rows[5:], **kw)                     # local indices: other streams
    assert local.out_tokens != whole.out_tokens[5:]
    with pytest.raises(ValueError):
        eng.generate(rows[5:], row_ids=[1, 2], **kw)


def test_one_call_c_entry_point_matches_the_phased_path():
    """sb200_infer_text (host buffers in/out, one C call) vs LocalEngine.generate."""
    spec, w, v, eng = build("tiny-qwen3", max_slots=8, max_prefill_tokens=512)
    rows = synth.product_reviews(19, seed=6) + ["", None]
    for kw in (dict(system_prompt=SYS, json_schema=SentimentEnum.model_json_schema(),
                    max_new_tokens=32),
               dict(system_prompt=SYS, max_new_tokens=9, ignore_eos=True),
               dict(max_new_tokens=12, temperature=0.8, top_k=30, seed=4, seed_per_row=True)):
        a = eng.generate(rows, return_tokens=True, return_logprobs=True, **kw)
        b = eng.infer_one_call(rows, return_logprobs=True, **kw)
        assert b.out_tokens == a.out_tokens and b.outputs == a.outputs
        assert np.allclose(b.cum_logprobs, a.cum_logprobs, atol=1e-4)
        assert b.stats["rows_done"] == len(rows)
    assert eng.infer_one_call([], max_new_tokens=4).outputs == []
    with pytest.raises(Exception):
        eng.infer_one_call(rows, max_new_tokens=0)


def test_one_call_c_entry_point_embedding_model():
    spec, w, v, eng = build("tiny-qwen3-embedding", max_slots=8, max_prefill_tokens=256)
    rows = synth.product_reviews(9, seed=2)
    a = eng.generate(rows)
    b = eng.infer_one_call(rows)
    assert np.array_equal(a.embeddings, b.embeddings)


def test_empty_and_null_inputs():
    spec, w, v, eng = build("tiny-qwen3", max_slots=4, max_prefill_tokens=256)
    assert eng.generate([], max_new_tokens=4).outputs == []
    res = eng.generate([None, "", "a"], max_new_tokens=2, ignore_eos=True, return_tokens=True)
    assert len(res.outputs) == 3 and all(len(t) == 2 for t in res.out_tokens)
    assert res.out_tokens[0] == res.out_tokens[1]        # null is the empty string


def test_embedding_model_matches_oracle():
    spec, w, v, eng = build("tiny-qwen3-embedding", max_slots=8, max_prefill_tokens=256)
    rows = synth.short_texts(20, seed=3)
    res = eng.generate(rows)
    assert res.embeddings.shape == (20, spec.d_model)
    ref_tok, model = RefTokenizer(v), RefModel(spec, w)
    tpl = VB.embedding_template(spec.family)
    for i, row in enumerate(rows):
        want = model.embed(ref_tok.render(tpl, row, spec.max_position)).numpy()
        assert np.abs(res.embeddings[i] - want).max() < EMB_TOL
        assert abs(np.linalg.norm(res.embeddings[i]) - 1.0) < 1e-3


def test_row_order_is_preserved_with_more_rows_than_slots():
    spec, w, v, eng = build("tiny-qwen3", max_slots=4, max_prefill_tokens=384, min_admit_rows=1)
    rows = synth.product_reviews(30, seed=5)
    res = eng.generate(rows, json_schema=SentimentEnum.model_json_schema(), max_new_tokens=32,
                       return_tokens=True)
    one_by_one = [eng.generate([r], json_schema=SentimentEnum.model_json_schema(),
                               max_new_tokens=32, return_tokens=True).out_tokens[0]
                  for r in rows[:10]]
    # batch-invariant kernels: a row decoded alone equals the same row decoded in a batch
    assert res.out_tokens[:10] == one_by_one
    assert res.stats["rows_done"] == 30 and res.stats["decode_steps"] > 0


@pytest.mark.parametrize("name", ["tiny-qwen3", "tiny-llama"])
def test_model_directory_on_disk_matches_oracle(name, tmp_path):
    """config.json + tokenizer.json (GPT-2 byte order, written by `tokenizers`) + safetensors ->
    pretrained.load_pretrained -> engine; the oracle runs on the checkpoint's own ids."""
    import json as _json

    from safetensors.torch import save_file

    import test_pretrained_cpu as TP
    from sutro_b200 import pretrained as PT
    spec = MS.get_spec(name)
    w = MS.make_weights(spec, seed=0, std=0.05)
    v = VB.build_vocab(spec.family, spec.vocab_size, seed=0, n_trained=600)
    hf = TP.gpt2_ordered_tokenizer(v)
    hf.save(str(tmp_path / "tokenizer.json"))
    (tmp_path / "config.json").write_text(_json.dumps(TP.hf_config(spec)))
    save_file({k: t.contiguous() for k, t in w.items()}, str(tmp_path / "model.safetensors"))
    eng = PT.load_pretrained(str(tmp_path), device=0, name=name, max_position=spec.max_position,
                             kv_pages=512, max_slots=8, max_prefill_tokens=512)
    loaded = eng.vocab
    assert loaded.id_map is not None and eng.spec == spec
    # a Qwen3 chat checkpoint is served the way its released template does it: the answer
    # opens with an empty think block, so the oracle's prompt carries one too
    assert eng.empty_think_block == (spec.family == "qwen3")
    res = eng.generate(ROWS, system_prompt=SYS, max_new_tokens=12, ignore_eos=True,
                       return_tokens=True)
    # oracle in the checkpoint's id space: tokenise with the loaded vocabulary, map to real ids
    ref_tok, model = RefTokenizer(loaded), RefModel(spec, w)
    tpl = VB.chat_template(spec.family, SYS, empty_think_block=eng.empty_think_block)
    real_eos = loaded.to_real_ids([loaded.eos_id])[0]
    compared = total = 0
    for row, got in zip(ROWS, res.out_tokens):
        prompt = loaded.to_real_ids(ref_tok.render(tpl, row, spec.max_position - 12))
        r = model.generate(prompt, 12, real_eos, ignore_eos=True)
        c, t, _ = compare_greedy(loaded.to_real_ids(got), r, row[:30], real_eos)
        compared, total = compared + c, total + t
    assert compared >= 0.5 * total, (compared, total)
