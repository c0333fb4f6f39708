"""The engine on the GQA-group-5 parity model (tiny-qwen3-g5: 10 q / 2 kv heads, q tile 25
tokens) end to end: greedy and schema-constrained decoding against the CPU oracle, batch
invariance, the paged prefill path against the tcgen05 one, a Hugging Face model directory on
disk and a model bundle served by the C host program."""
import json
import subprocess

import pytest

import test_c_host_gpu as TC
import test_engine_gpu as TE
from oracle.bpe_ref import RefTokenizer
from oracle.fsm_ref import TokenFSM
from oracle.model_ref import RefModel
from sutro_b200 import modelspec as MS
from sutro_b200 import synth, vocab as VB
from sutro_b200.schema_fsm import FsmLimits, compile_schema

pytestmark = pytest.mark.gpu

NAME = "tiny-qwen3-g5"


def test_unconstrained_greedy_matches_oracle_group5():
    TE.test_unconstrained_greedy_matches_oracle(NAME)


def test_teacher_forced_logits_within_tolerance_group5():
    TE.test_teacher_forced_logits_within_tolerance(NAME)


def test_schema_outputs_validate_and_match_oracle_group5():
    spec, w, v, eng = TE.build(NAME, max_slots=8, max_prefill_tokens=512)
    schema = TE.SentimentEnum.model_json_schema()
    res = eng.generate(TE.ROWS, system_prompt=TE.SYS, json_schema=schema, max_new_tokens=32,
                       return_tokens=True)
    dfa = compile_schema(schema, FsmLimits())
    fsm = TokenFSM(dfa, v)
    ref_tok, model = RefTokenizer(v), RefModel(spec, w)
    assert fsm.enable_jump_forward(ref_tok)
    tpl = VB.chat_template(spec.family, TE.SYS)
    compared = total = flips = 0
    for row, text, got in zip(TE.ROWS, res.outputs, res.out_tokens):
        TE.SentimentEnum.model_validate(json.loads(text))
        r = model.generate(ref_tok.render(tpl, row), 32, v.eos_id, fsm=fsm)
        c, t, f = TE.compare_greedy(got, r, row[:30], v.eos_id)
        compared, total, flips = compared + c, total + t, flips + f
    TE.record_parity(f"schema[SentimentEnum,{NAME}]", len(TE.ROWS), compared, total, flips)
    assert compared >= 0.5 * total, (compared, total)
    assert flips <= TE.MAX_FLIP_ROWS, flips


def test_a_row_alone_equals_the_row_in_a_batch_group5():
    spec, w, v, eng = TE.build(NAME, max_slots=4, max_prefill_tokens=384, min_admit_rows=1)
    rows = synth.product_reviews(24, seed=5) + TE.ROWS[-3:]
    res = eng.generate(rows, system_prompt=TE.SYS, max_new_tokens=8, ignore_eos=True,
                       return_tokens=True)
    for i in (0, 3, 7, 24, 26):
        alone = eng.generate([rows[i]], system_prompt=TE.SYS, max_new_tokens=8, ignore_eos=True,
                             return_tokens=True).out_tokens[0]
        assert alone == res.out_tokens[i], i


def test_paged_prefill_path_gives_the_tcgen05_tokens_group5(monkeypatch):
    rows = synth.product_reviews(20, seed=13) + TE.ROWS
    kw = dict(system_prompt=TE.SYS, max_new_tokens=8, ignore_eos=True, return_tokens=True)
    spec, w, v, eng = TE.build(NAME, max_slots=16, max_prefill_tokens=1024)
    tc = eng.generate(rows, **kw).out_tokens
    eng.close()
    monkeypatch.setenv("SB200_PREFILL_TC", "0")     # read when the engine is created
    _, _, _, eng = TE.build(NAME, max_slots=16, max_prefill_tokens=1024)
    paged = eng.generate(rows, **kw).out_tokens
    eng.close()
    # two kernels, two fp32 summation orders: where the tokens differ, the paged path's must
    # still be the oracle's up to a near-tie flip
    ref_tok, model = RefTokenizer(v), RefModel(spec, w)
    tpl = VB.chat_template(spec.family, TE.SYS)
    same = 0
    for row, a, b in zip(rows, tc, paged):
        same += a == b
        if a != b:
            r = model.generate(ref_tok.render(tpl, row), 8, v.eos_id, ignore_eos=True)
            TE.compare_greedy(b, r, row[:30], v.eos_id)
    TE.record_parity(f"paged_vs_tcgen05_prefill[{NAME}]", len(rows), same, len(rows), 0)
    assert same >= len(rows) - 3, (same, len(rows))


def test_model_directory_on_disk_matches_oracle_group5(tmp_path):
    TE.test_model_directory_on_disk_matches_oracle(NAME, tmp_path)


def test_c_program_matches_the_python_host_group5(tmp_path):
    """As test_c_host_gpu.py; the unconstrained run uses the C host's default output budget
    (512 tokens, capped at half of this model's 1024-token window) on both sides."""
    from sutro_b200.bundle import export_bundle
    from sutro_b200.engine import LocalEngine
    exe = TC._compile(tmp_path)
    spec = MS.get_spec(NAME)
    w = MS.make_weights(spec, seed=0, std=0.05)
    v = VB.build_vocab(spec.family, spec.vocab_size, seed=0, n_trained=600)
    eng = LocalEngine(spec, MS.pack_for_engine(spec, w, "cuda"), v, device=0, kv_pages=512,
                      max_slots=8, max_prefill_tokens=512)
    bundle = export_bundle(eng, str(tmp_path / "bundle"))
    schema = TC.Sentiment.model_json_schema()
    (tmp_path / "schema.json").write_text(json.dumps(schema))
    rows = synth.README_REVIEWS + ["", "café naïve 東京"]
    want = eng.generate(rows, system_prompt=synth.README_SYSTEM_PROMPT, json_schema=schema,
                        max_new_tokens=len('{"sentiment":"positive"}')).outputs
    free = eng.generate(rows, system_prompt=None,
                        max_new_tokens=min(512, spec.max_position // 2)).outputs
    eng.close()
    out = subprocess.run([exe, bundle, synth.README_SYSTEM_PROMPT, str(tmp_path / "schema.json")]
                         + rows, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    got = out.stdout.split("\n")[:len(rows)]
    assert got == want, (got, want, out.stderr[-500:])
    for text in got:
        TC.Sentiment.model_validate(json.loads(text))
    out = subprocess.run([exe, bundle, "", "-"] + rows, capture_output=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    got = out.stdout.decode("utf-8", errors="replace").split("\n")
    assert got[0] == free[0].split("\n")[0]
