"""The drop-in call itself on hardware: `sutro_b200.infer(df, column=, model=, system_prompt=,
output_schema=)` -> `get_job_results(job_id, with_original_df=df)` as in the reference's README
(README.md:33-56) and `Sutro.infer` / `get_job_results` (sutro/sdk.py:434-502, :1037-1190,
:1172-1184) — SDK layer, C-ABI and engine together, no stub anywhere."""
import json
from typing import Literal

import numpy as np
import pandas as pd
import pytest
from pydantic import BaseModel

from sutro_b200 import synth

pytestmark = pytest.mark.gpu


class Sentiment(BaseModel):           # README.md:45-46 with the label set of tests/test_sdk.py:427-435
    sentiment: Literal["positive", "neutral", "negative"]


class FreeSentiment(BaseModel):       # README.md:45-46 verbatim: a free string
    sentiment: str


OPTS = dict(kv_pages=512, max_slots=8, max_prefill_tokens=512)


def test_readme_flow_through_the_module_level_api(tmp_path):
    import sutro_b200 as so
    client = so.configure(engine_options=OPTS, verbose=False, cache_dir=str(tmp_path))
    df = pd.DataFrame({"review": synth.README_REVIEWS, "id": [7, 8, 9]})
    job_id = so.infer(df, column="review", model="tiny-qwen3",
                      system_prompt=synth.README_SYSTEM_PROMPT, output_schema=Sentiment)
    assert isinstance(job_id, str) and so.get_job_status(job_id) == so.JobStatus.SUCCEEDED
    # attached p0 job: the pandas frame is updated in place (sutro/sdk.py:408-412)
    assert list(df.columns) == ["review", "id", "inference_result"]
    for text in df["inference_result"]:
        Sentiment.model_validate(json.loads(text))
    res = so.get_job_results(job_id, with_original_df=df, include_inputs=True)
    assert list(res["review"]) == synth.README_REVIEWS and list(res["id"]) == [7, 8, 9]
    assert list(res["inputs"]) == synth.README_REVIEWS
    assert list(res["sentiment"]) == [json.loads(t)["sentiment"] for t in df["inference_result"]]
    assert "confidence_score" in res.columns and all(0 < c <= 1.0 + 1e-6 for c in res["confidence_score"])
    # the same rows through the engine directly: the SDK adds plumbing, not arithmetic
    eng = client._engine("tiny-qwen3")
    direct = eng.generate(synth.README_REVIEWS, system_prompt=synth.README_SYSTEM_PROMPT,
                          json_schema=Sentiment.model_json_schema(),
                          max_new_tokens=len('{"sentiment":"positive"}'))
    assert direct.outputs == list(df["inference_result"])
    # detached job + await_job_completion, list input, free-string schema, more rows than slots
    rows = synth.product_reviews(21, seed=3)
    job2 = so.infer(rows, model="tiny-qwen3", system_prompt=synth.README_SYSTEM_PROMPT,
                    output_schema=FreeSentiment, job_priority=1,
                    sampling_params={"max_tokens": 40})
    out = so.await_job_completion(job2)
    assert len(out) == 21
    # rows cut by max_tokens are not JSON: they unpack to nulls, the rest validate
    ok = 0
    for text, val in zip(so.get_job_results(job2, unpack_json=False)["inference_result"],
                         out["sentiment"]):
        try:
            FreeSentiment.model_validate(json.loads(text))
            ok += 1
        except ValueError:
            assert pd.isna(val)
    assert ok >= 1


def test_templates_run_on_the_real_engine(tmp_path):
    """classify / score / embed (sutro/templates/*.py call infer + await_job_completion)."""
    import sutro_b200 as so
    so.configure(engine_options=OPTS, verbose=False, cache_dir=str(tmp_path))
    df = pd.DataFrame({"text": synth.product_reviews(6, seed=1)})
    cls = so.classify(df, ["good", "bad", "mixed"], model="tiny-qwen3", column="text")
    assert len(cls) == 6 and set(cls["inference_result"]) <= {"good", "bad", "mixed"}
    sc = so.score(df, model="tiny-qwen3", column="text", criteria="clarity", range=(1, 5))
    assert list(sc.columns) == ["text", "score"] and all(1 <= int(x) <= 5 for x in sc["score"])
    emb = so.embed(df, model="tiny-qwen3-embedding", column="text")
    vecs = np.stack([np.asarray(v) for v in emb["inference_result"]])
    assert vecs.shape[0] == 6 and np.allclose(np.linalg.norm(vecs, axis=1), 1.0, atol=1e-3)


def test_thinking_model_outputs_content_and_reasoning(tmp_path):
    """"<model>-thinking": reasoning first (capped), then the schema-constrained answer; the
    job reports {"content", "reasoning_content"} (sutro/sdk.py:1155-1164, common.py:28-32)."""
    import sutro_b200 as so
    so.configure(engine_options=OPTS, verbose=False, cache_dir=str(tmp_path))
    rows = synth.README_REVIEWS + synth.product_reviews(5, seed=8)
    job = so.infer(rows, model="tiny-qwen3-thinking", system_prompt=synth.README_SYSTEM_PROMPT,
                   output_schema=Sentiment, sampling_params={"max_thinking_chars": 24},
                   stay_attached=False)
    raw = so.get_job_results(job, unpack_json=False)["inference_result"]
    for text in raw:
        obj = json.loads(text)
        assert sorted(obj) == ["content", "reasoning_content"]
        Sentiment.model_validate(obj["content"])
        assert len(obj["reasoning_content"]) <= 24 and "<" not in obj["reasoning_content"]
    df = so.get_job_results(job)
    assert set(df["sentiment"]) <= {"positive", "neutral", "negative"}
    assert "reasoning_content" in df.columns and "content" not in df.columns


def test_arrow_helpers_match_numpy():
    """sb200_rows_select / sb200_compact_rows (the kernels behind row sharding, the ordered
    gather and output compaction) against numpy — bit-exact."""
    import torch

    from sutro_b200 import _lib as L
    from sutro_b200 import engine as E
    rng = np.random.RandomState(0)
    rows = ["", "a", "héllo"] + ["x" * int(k) for k in rng.randint(0, 300, size=500)]
    data, off = E.rows_to_blob(rows)
    d_b = torch.from_numpy(np.ascontiguousarray(data)).cuda()
    d_o = torch.from_numpy(np.ascontiguousarray(off)).cuda()
    idx = rng.permutation(len(rows))[:200].astype(np.int64)
    d_idx = torch.from_numpy(idx).cuda()
    o_off = torch.empty(len(idx) + 1, dtype=torch.int64, device="cuda")
    o_b = torch.zeros(max(len(data), 1), dtype=torch.uint8, device="cuda")
    L.check(L.lib().sb200_rows_select(d_b.data_ptr(), d_o.data_ptr(), len(rows), 0,
                                      d_idx.data_ptr(), len(idx), o_off.data_ptr(),
                                      o_b.data_ptr(), L.current_stream()))
    got = E.blob_to_rows(o_b.cpu().numpy(), o_off.cpu().numpy())
    assert got == [rows[i] for i in idx]
    # batch of two equally strided parts (what the NCCL gather of padded results looks like)
    parts = [["p0r0", "p0-row1", ""], ["q", "qq", "qqq"]]
    blobs = [E.rows_to_blob(p) for p in parts]
    max_b = max(len(b) for b, _ in blobs)
    pb = np.zeros((2, max_b), np.uint8)
    po = np.zeros((2, 4), np.int64)
    for k, (b, o) in enumerate(blobs):
        pb[k, :len(b)] = b
        po[k] = o
    sel = np.array([3, 0, 5, 1, 4, 2], dtype=np.int64)     # row j -> part j // 3, local j % 3
    d_pb, d_po, d_sel = (torch.from_numpy(x).cuda() for x in (pb.reshape(-1), po.reshape(-1), sel))
    m_off = torch.empty(7, dtype=torch.int64, device="cuda")
    m_b = torch.zeros(2 * max_b, dtype=torch.uint8, device="cuda")
    L.check(L.lib().sb200_rows_select(d_pb.data_ptr(), d_po.data_ptr(), 3, max_b,
                                      d_sel.data_ptr(), 6, m_off.data_ptr(), m_b.data_ptr(),
                                      L.current_stream()))
    flat = [r for p in parts for r in p]
    assert E.blob_to_rows(m_b.cpu().numpy(), m_off.cpu().numpy()) == [flat[j] for j in sel]
    # compaction
    n, stride = 300, 9
    toks = torch.from_numpy(rng.randint(0, 1000, size=(n, stride)).astype(np.int32)).cuda()
    lens = torch.from_numpy(rng.randint(0, stride + 1, size=n).astype(np.int32)).cuda()
    c_off = torch.empty(n + 1, dtype=torch.int64, device="cuda")
    c_flat = torch.zeros(n * stride, dtype=torch.int32, device="cuda")
    L.check(L.lib().sb200_compact_rows(toks.data_ptr(), lens.data_ptr(), n, stride,
                                       c_off.data_ptr(), c_flat.data_ptr(), L.current_stream()))
    ln = lens.cpu().numpy()
    want_off = np.concatenate([[0], np.cumsum(ln)])
    assert np.array_equal(c_off.cpu().numpy(), want_off)
    want = np.concatenate([toks.cpu().numpy()[i, :ln[i]] for i in range(n)])
    assert np.array_equal(c_flat.cpu().numpy()[:len(want)], want)
