"""Qwen3-14B and Qwen3-32B at their real widths (d_model 5120; 40 / 8 and 64 / 8 heads; d_ff
17408 / 25600) on seeded random weights.

Parity: the real geometry truncated in depth (4 layers of 14B, 3 of 32B: the CPU oracle has
to multiply them on the host), first-decision logits against the bf16 and the exact oracle
under the noise-floor criterion of test_zy_real_size_parity_gpu.py.  Serving: the full-depth
qwen-3-14b through the SDK with a schema, plain and as "-thinking".  The file name sorts it
near the end of the suite."""
import json
import os
from dataclasses import replace
from typing import Literal

import pytest
import torch
from pydantic import BaseModel

import test_zy_real_size_parity_gpu as RS
from oracle.bpe_ref import RefTokenizer
from oracle.model_ref import RefModel
from sutro_b200 import modelspec as MS
from sutro_b200 import synth, vocab as VB

pytestmark = pytest.mark.gpu


class Sentiment(BaseModel):
    sentiment: Literal["positive", "neutral", "negative"]


@pytest.mark.parametrize("name,layers", [("qwen-3-14b", 4), ("qwen-3-32b", 3)])
def test_first_decision_logits_match_the_oracle_at_real_width(name, layers):
    from sutro_b200.engine import LocalEngine
    torch.set_num_threads(min(64, os.cpu_count() or 1))
    spec = replace(MS.get_spec(name), n_layers=layers)
    w = MS.make_engine_weights_on_device(spec, 0, "cuda")
    v = VB.build_vocab(spec.family, spec.vocab_size, seed=0)
    eng = LocalEngine(spec, w, v, device=0, kv_pages=2048, max_slots=16, max_prefill_tokens=4096)
    try:
        res = eng.generate(RS.ROWS, system_prompt=RS.SYS, max_new_tokens=1, ignore_eos=True,
                           return_tokens=True, return_first_logits=True)
        model, tok = RefModel(spec, MS.unpack_to_hf(spec, w), fast=True), RefTokenizer(v)
        tpl = VB.chat_template(spec.family, RS.SYS)
        worst_rms = worst_max = 0.0
        agree = 0
        noise_eng, noise_orc = [], []
        for i, row in enumerate(RS.ROWS):
            prompt = tok.render(tpl, row)
            want = model.logits(prompt)[-1]
            got = res.first_logits[i]
            sd = want.std().item()
            d = (got - want).abs()
            rms, mx = d.pow(2).mean().sqrt().item() / sd, d.max().item() / sd
            worst_rms, worst_max = max(worst_rms, rms), max(worst_max, mx)
            if i < 2:
                exact = model.logits(prompt, exact=True)[-1]
                noise_eng.append((got - exact).pow(2).mean().sqrt().item() / sd)
                noise_orc.append((want - exact).pow(2).mean().sqrt().item() / sd)
            top2 = torch.topk(want, 2).values
            margin = (top2[0] - top2[1]).item()
            same = int(got.argmax()) == int(want.argmax())
            agree += same
            assert same or margin < 0.06, (name, i, margin)
            assert res.out_tokens[i][0] == int(got.argmax())
        RS._record({"model": f"{name}[{layers} layers]", "rows": len(RS.ROWS),
                    "logit_rms_over_sigma": worst_rms, "logit_max_over_sigma": worst_max,
                    "argmax_equal": f"{agree}/{len(RS.ROWS)}", "rms_engine_vs_exact": noise_eng,
                    "rms_bf16_oracle_vs_exact": noise_orc})
        assert worst_rms < RS.RMS_TOL and worst_max < RS.MAX_TOL, (worst_rms, worst_max)
        for e, o in zip(noise_eng, noise_orc):
            assert e <= RS.NOISE_FACTOR * o + RS.NOISE_SLACK, (e, o)
    finally:
        eng.close()
        del eng, w
        torch.cuda.empty_cache()


def test_qwen3_14b_serves_schema_jobs_through_the_sdk(tmp_path):
    import sutro_b200 as so
    client = so.Sutro(engine_options=dict(kv_pages=4096, max_slots=64, max_prefill_tokens=4096),
                      verbose=False, cache_dir=str(tmp_path))
    rows = synth.README_REVIEWS + synth.product_reviews(13, seed=4)
    try:
        job = client.infer(rows, model="qwen-3-14b", system_prompt=synth.README_SYSTEM_PROMPT,
                           output_schema=Sentiment, stay_attached=False)
        raw = client.get_job_results(job, unpack_json=False)["inference_result"]
        assert len(raw) == len(rows)
        for text in raw:
            Sentiment.model_validate(json.loads(text))
        job = client.infer(rows[:6], model="qwen-3-14b-thinking",
                           system_prompt=synth.README_SYSTEM_PROMPT, output_schema=Sentiment,
                           sampling_params={"max_thinking_chars": 24}, stay_attached=False)
        raw = client.get_job_results(job, unpack_json=False)["inference_result"]
        assert len(raw) == 6
        for text in raw:
            obj = json.loads(text)
            assert sorted(obj) == ["content", "reasoning_content"]
            Sentiment.model_validate(obj["content"])
        assert list(client._engines) == ["qwen-3-14b"]       # "-thinking": the same weights
    finally:
        for eng in client._engines.values():
            eng.close()
        client._engines.clear()
        torch.cuda.empty_cache()
