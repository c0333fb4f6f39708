"""CPU tests of the drop-in boundary: argument handling, error conventions and result
shaping follow the reference (sutro/common.py:72-163, sutro/sdk.py:186-193, :406-432,
:1111-1170; reference tests/test_sdk.py:326-334).  The engine is replaced by a stub —
these tests are about the host logic only."""
import inspect
import json
import os
import tempfile

import numpy as np
import pandas as pd
import pytest
from pydantic import BaseModel

import sutro_b200 as so
from sutro_b200 import common, interfaces
from sutro_b200.engine import GenerationResult, rows_to_blob, blob_to_rows
from sutro_b200.sdk import Sutro


# the clients' results cache: private to this run (a fixed path under /tmp may belong to
# another user of the machine)
_CACHE = tempfile.TemporaryDirectory(prefix="sb200-test-cache-")
CACHE = _CACHE.name


class Sentiment(BaseModel):
    sentiment: str


class StubEngine:
    def __init__(self, as_json=True):
        self.calls, self.as_json = [], as_json

    def generate(self, rows, **kw):
        self.calls.append((list(rows), kw))
        outs = [json.dumps({"sentiment": f"s{i}"}) if self.as_json else f"out-{i}"
                for i in range(len(rows))]
        return GenerationResult(outs, None, None, {"input_tokens": 10, "output_tokens": 5})


def client(as_json=True):
    c = Sutro(verbose=False, cache_dir=CACHE)
    c.register_engine("qwen-3-4b", StubEngine(as_json))
    return c


def test_infer_signature_matches_reference_positional_order():
    want = ["self", "data", "model", "name", "description", "column", "output_column",
            "job_priority", "output_schema", "sampling_params", "system_prompt", "dry_run",
            "stay_attached", "random_seed_per_input", "truncate_rows"]
    assert list(inspect.signature(Sutro.infer).parameters) == want
    assert list(inspect.signature(interfaces.BaseSutroClient.infer).parameters) == want
    p = inspect.signature(Sutro.infer).parameters
    assert p["model"].default == "gemma-3-12b-it" and p["output_column"].default == "inference_result"
    assert p["job_priority"].default == 0 and p["truncate_rows"].default is True
    assert list(inspect.signature(Sutro.await_job_completion).parameters) == [
        "self", "job_id", "timeout", "obtain_results", "output_column", "is_cost_estimate"]
    assert callable(so.infer) and callable(so.get_job_results)


def test_job_status_enum_matches_reference():
    names = ["UNKNOWN", "QUEUED", "STARTING", "RUNNING", "SUCCEEDED", "CANCELLING", "CANCELLED",
             "FAILED"]
    assert [s.name for s in interfaces.JobStatus] == names
    assert interfaces.JobStatus.SUCCEEDED.is_terminal() and not interfaces.JobStatus.RUNNING.is_terminal()


def test_missing_column_raises_value_error():           # reference tests/test_sdk.py:326-334
    with pytest.raises(ValueError, match="Column name must be specified"):
        client().infer(pd.DataFrame({"a": ["x"]}), model="qwen-3-4b")


def test_name_and_description_limits():                  # sutro/sdk.py:186-193
    with pytest.raises(ValueError, match="Job name cannot exceed 45"):
        client().infer(["x"], model="qwen-3-4b", name="n" * 46)
    with pytest.raises(ValueError, match="description cannot exceed 512"):
        client().infer(["x"], model="qwen-3-4b", description="d" * 513)


def test_invalid_schema_raises_value_error():            # sutro/common.py:161-163
    with pytest.raises(ValueError, match="Invalid output schema type"):
        client().infer(["x"], model="qwen-3-4b", output_schema="nope")
    assert common.normalize_output_schema(Sentiment)["properties"]["sentiment"]["type"] == "string"
    assert common.normalize_output_schema({"type": "object"}) == {"type": "object"}


def test_column_concatenation_with_literal_separators():  # sutro/common.py:72-108
    df = pd.DataFrame({"a": ["x", None], "b": [1, 2]})
    assert common.handle_data_helper(df, ["a", ": ", "b"]) == ["x: 1", ": 2"]
    assert common.handle_data_helper(df, "b") == [1, 2]
    assert common.handle_data_helper(["p", "q"]) == ["p", "q"]
    with pytest.raises(ValueError, match="Unsupported data type"):
        common.handle_data_helper(42)


def test_attached_pandas_is_updated_in_place_and_job_id_returned():   # sutro/sdk.py:406-430
    c = client()
    df = pd.DataFrame({"review": ["a", "b", "c"]})
    job_id = c.infer(df, model="qwen-3-4b", column="review", output_schema=Sentiment,
                     system_prompt="classify")
    assert isinstance(job_id, str) and job_id.startswith("job-")
    assert list(df["inference_result"]) == [json.dumps({"sentiment": f"s{i}"}) for i in range(3)]
    eng = c._engines["qwen-3-4b"]
    rows, kw = eng.calls[0]
    assert rows == ["a", "b", "c"] and kw["system_prompt"] == "classify"
    assert kw["json_schema"]["properties"]["sentiment"]["type"] == "string"
    assert c.get_job_status(job_id) == interfaces.JobStatus.SUCCEEDED


def test_detached_returns_job_id_and_results_are_unpacked():   # sdk.py:256-273, :1137-1154
    c = client()
    df = pd.DataFrame({"review": ["a", "b"]})
    job_id = c.infer(df, model="qwen-3-4b", column="review", job_priority=1)
    assert "inference_result" not in df.columns           # detached: no write-back
    res = c.await_job_completion(job_id)
    assert list(res.columns) == ["sentiment"] and list(res["sentiment"]) == ["s0", "s1"]
    joined = c.get_job_results(job_id, with_original_df=df, include_inputs=True)
    assert list(joined.columns) == ["review", "inputs", "sentiment"]
    raw = c.get_job_results(job_id, unpack_json=False, output_column="out")
    assert list(raw.columns) == ["out"]


def test_plain_text_outputs_are_not_unpacked():
    c = client(as_json=False)
    job_id = c.infer(["a", "b"], model="qwen-3-4b", stay_attached=False)
    res = c.get_job_results(job_id)
    assert list(res.columns) == ["inference_result"] and list(res["inference_result"]) == ["out-0", "out-1"]


def test_engine_failure_prints_and_returns_none():        # non-200 convention, sdk.py:225-234
    c = Sutro(verbose=False)

    class Boom:
        def generate(self, rows, **kw):
            raise RuntimeError("device lost")
    c.register_engine("qwen-3-4b", Boom())
    assert c.infer(["x"], model="qwen-3-4b") is None
    assert c.list_jobs()[0]["status"] == "FAILED"


def test_sampling_params_are_mapped_and_unknown_keys_rejected():
    c = client()
    c.infer(["x"], model="qwen-3-4b", sampling_params={"temperature": 0.7, "top_p": 0.9,
                                                        "top_k": 40, "seed": 5, "max_tokens": 12},
            random_seed_per_input=True)
    kw = c._engines["qwen-3-4b"].calls[0][1]
    assert (kw["temperature"], kw["top_p"], kw["top_k"], kw["seed"], kw["max_new_tokens"]) == \
        (0.7, 0.9, 40, 5, 12)
    assert kw["seed_per_row"] is True
    with pytest.raises(ValueError, match="unsupported sampling_params"):
        client().infer(["x"], model="qwen-3-4b", sampling_params={"beam_width": 4})
    with pytest.raises(ValueError, match="top_p"):
        client().infer(["x"], model="qwen-3-4b", sampling_params={"top_p": 0})


def test_cumulative_logprobs_column():
    c = Sutro(verbose=False, cache_dir=CACHE)

    class E:
        def generate(self, rows, **kw):
            return GenerationResult([f"o{i}" for i in range(len(rows))], None, None, {},
                                    None, np.array([-1.5, -0.25], dtype=np.float32))
    c.register_engine("qwen-3-4b", E())
    jid = c.infer(["a", "b"], model="qwen-3-4b", stay_attached=False)
    df = c.get_job_results(jid, include_cumulative_logprobs=True, include_inputs=True)
    assert list(df.columns) == ["inputs", "inference_result", "cumulative_logprobs"]
    assert list(df["cumulative_logprobs"]) == [-1.5, -0.25]


def test_infer_per_model_returns_list_of_ids():           # sutro/sdk.py:750-757
    c = client()
    c.register_engine("m2", StubEngine())
    ids = c.infer_per_model(["x"], ["qwen-3-4b", "m2"])
    assert len(ids) == 2 and all(i.startswith("job-") for i in ids)


def test_rows_to_blob_roundtrip_arrow_style():
    rows = ["héllo", "", None, "x" * 1000, "日本"]
    data, off = rows_to_blob(rows)
    assert off.dtype == np.int64 and len(off) == 6 and off[0] == 0
    assert blob_to_rows(data, off) == ["héllo", "", "", "x" * 1000, "日本"]
    import pyarrow as pa
    d2, o2 = rows_to_blob(pa.array(["a", "bc"]).slice(1))
    assert blob_to_rows(d2, o2) == ["bc"]


# --------------------------------------------------------------------------- templates
class SchemaEcho:
    """Stub engine that answers according to the schema it was given."""
    def __init__(self):
        self.calls = []

    def generate(self, rows, **kw):
        self.calls.append((list(rows), kw))
        props = (kw.get("json_schema") or {}).get("properties", {})
        outs = []
        for i, _ in enumerate(rows):
            obj = {}
            for k, sch in props.items():
                if "enum" in sch:
                    obj[k] = sch["enum"][i % len(sch["enum"])]
                elif sch.get("type") == "array":
                    obj[k] = list(sch["items"]["enum"])[: sch["minItems"]]
                elif sch.get("type") == "integer":
                    obj[k] = sch["minimum"] + i % (sch["maximum"] - sch["minimum"] + 1)
                else:
                    obj[k] = f"t{i}"
            outs.append(json.dumps(obj))
        return GenerationResult(outs, None, None, {})


def test_template_signatures_match_reference():
    assert list(inspect.signature(Sutro.classify).parameters) == [
        "self", "data", "classes", "model", "job_priority", "name", "description",
        "output_column", "column", "truncate_rows", "include_scratchpad"]
    assert list(inspect.signature(Sutro.embed).parameters) == [
        "self", "data", "model", "job_priority", "name", "description", "output_column",
        "column", "truncate_rows"]
    assert list(inspect.signature(Sutro.score).parameters) == [
        "self", "data", "model", "job_priority", "name", "description", "column", "criteria",
        "score_column_name", "range"]
    assert inspect.signature(Sutro.embed).parameters["model"].default == "qwen-3-embedding-0.6b"


def test_classify_constrains_to_the_label_set():
    c = Sutro(verbose=False, cache_dir=CACHE)
    eng = SchemaEcho()
    c.register_engine("m", eng)
    df = pd.DataFrame({"t": ["a", "b", "c"]})
    out = c.classify(df, {"pos": "happy", "neg": "unhappy"}, model="m", column="t")
    assert list(out.columns) == ["inference_result"] and list(out["inference_result"]) == ["pos", "neg", "pos"]
    kw = eng.calls[0][1]
    assert kw["json_schema"]["properties"]["classification"]["enum"] == ["pos", "neg"]
    assert "happy" in kw["system_prompt"]
    full = c.classify(df, ["x", "y"], model="m", column="t", include_scratchpad=True)
    assert list(full.columns) == ["scratchpad", "classification"]
    with pytest.raises(ValueError):
        c.classify(df, [], model="m", column="t")


def test_score_appends_bounded_integer_column():
    c = Sutro(verbose=False, cache_dir=CACHE)
    eng = SchemaEcho()
    c.register_engine("m", eng)
    df = pd.DataFrame({"t": ["a", "b", "c"]})
    out = c.score(df, model="m", column="t", criteria=["clarity", "tone"], range=(1, 5),
                  score_column_name="s")
    assert list(out.columns) == ["t", "s"] and list(out["s"]) == [1, 2, 3]
    sch = eng.calls[0][1]["json_schema"]["properties"]["s"]
    assert (sch["minimum"], sch["maximum"]) == (1, 5)
    assert "t" in df.columns and "s" not in df.columns       # input frame is not mutated
    with pytest.raises(ValueError):
        c.score(df, model="m", column="t")


def test_embed_returns_vector_column():
    c = Sutro(verbose=False, cache_dir=CACHE)

    class Emb:
        def generate(self, rows, **kw):
            return GenerationResult(None, None, np.eye(len(rows), 4, dtype=np.float32), {})
    c.register_engine("qwen-3-embedding-0.6b", Emb())
    out = c.embed(["a", "b"])
    assert list(out.columns) == ["inference_result"]
    assert out["inference_result"][1].tolist() == [0, 1, 0, 0]
    import pyarrow.parquet as pq
    jid = c.list_jobs()[-1]["job_id"]
    t = pq.read_table(os.path.join(CACHE, f"{jid}.snappy.parquet"))
    assert t.column("inference_result").to_pylist()[1] == [0.0, 1.0, 0.0, 0.0]
    assert c.get_job_embeddings(jid).shape == (2, 4)


def test_rank_returns_permutations_and_prints_elo(capsys):
    c = Sutro(verbose=False, cache_dir=CACHE)
    eng = SchemaEcho()
    c.register_engine("m", eng)
    assert list(inspect.signature(Sutro.rank).parameters) == [
        "self", "model", "job_priority", "name", "description", "data", "option_labels",
        "criteria", "ranking_column_name", "run_elo"]            # sutro/templates/evals.py:78-93
    assert list(inspect.signature(Sutro.elo).parameters) == [
        "data", "column", "laplace", "max_iter", "tol", "elo_mean"]
    rows = [["short", "long", "mid"], ["x", None, "z"], ["1", "2", "3"], ["q", "r", "s"]]
    out = c.rank(model="m", data=rows, option_labels=["A", "B", "C"], criteria="brevity")
    assert list(out.columns) == ["A", "B", "C", "ranking"]
    assert all(sorted(r) == ["A", "B", "C"] for r in out["ranking"])
    sent, kw = eng.calls[0]
    assert sent[0] == "A: short B: long C: mid" and sent[1] == "A: x B:  C: z"
    perms = kw["json_schema"]["properties"]["ranking"]["enum"]
    assert len(perms) == 6 and ["B", "A", "C"] in perms
    assert "brevity" in kw["system_prompt"]
    assert "elo" in capsys.readouterr().out
    # pandas frame in -> pandas frame out with the ranking appended; input not mutated
    df = pd.DataFrame({"A": ["a1", "a2"], "B": ["b1", "b2"], "other": [1, 2]})
    out2 = c.rank(model="m", data=df, option_labels=["B", "A"], criteria=["c1", "c2"],
                  ranking_column_name="order", run_elo=False)
    assert list(out2.columns) == ["A", "B", "other", "order"] and "order" not in df.columns
    assert eng.calls[-1][0][0] == "B: b1 A: a1"
    # more than six labels: array-of-enum schema with a fixed length
    labels = [f"L{i}" for i in range(7)]
    c.rank(model="m", data=[[str(i) for i in range(7)]], option_labels=labels, criteria="x",
           run_elo=False)
    assert eng.calls[-1][1]["json_schema"]["properties"]["ranking"]["minItems"] == 7
    with pytest.raises(ValueError):
        c.rank(model="m", data=[["only-one"]], option_labels=["A", "B"], criteria="x")
    with pytest.raises(ValueError):
        c.rank(model="m", data=df, option_labels=["A", "missing"], criteria="x")
    with pytest.raises(ValueError):
        c.rank(model="m", data=df, option_labels=["A", "A"], criteria="x")


def test_rank_schemas_compile_to_permutation_dfas():
    """The rank schemas are inside the FSM compiler's subset; the small-n one admits exactly
    the permutations."""
    import itertools
    from sutro_b200.schema_fsm import compile_schema
    labels = ["A", "B", "C"]
    sch = {"type": "object", "properties": {"ranking": {"enum": [list(p) for p in
                                                                  itertools.permutations(labels)]}},
           "required": ["ranking"]}
    dfa = compile_schema(sch)
    assert dfa.matches(b'{"ranking":["B","A","C"]}')
    assert not dfa.matches(b'{"ranking":["B","B","C"]}')
    assert not dfa.matches(b'{"ranking":["B","A"]}')
    big = [f"L{i}" for i in range(7)]
    sch7 = {"type": "object", "properties": {"ranking": {"type": "array", "items": {
        "type": "string", "enum": big}, "minItems": 7, "maxItems": 7}}, "required": ["ranking"]}
    dfa7 = compile_schema(sch7)
    assert dfa7.matches(('{"ranking":' + json.dumps(big, separators=(",", ":")) + "}").encode())
    assert not dfa7.matches(('{"ranking":' + json.dumps(big[:6], separators=(",", ":")) + "}").encode())


def test_confidence_score_column_for_schema_jobs():
    c = Sutro(verbose=False, cache_dir=CACHE)

    class E:
        def generate(self, rows, **kw):
            outs = [json.dumps({"sentiment": "pos"}) for _ in rows]
            return GenerationResult(outs, None, None, {}, None,
                                    np.log(np.array([0.5, 0.25], dtype=np.float32)))
    c.register_engine("qwen-3-4b", E())
    jid = c.infer(["a", "b"], model="qwen-3-4b", output_schema=Sentiment, stay_attached=False)
    df = c.get_job_results(jid, include_cumulative_logprobs=True)
    assert list(df.columns) == ["cumulative_logprobs", "confidence_score", "sentiment"]
    assert np.allclose(df["confidence_score"], [0.5, 0.25])
    raw = c.get_job_results(jid, unpack_json=False)
    assert list(raw.columns) == ["inference_result", "confidence_score"]
    # no schema -> no confidence column (only cumulative logprobs on request)
    jid2 = c.infer(["a", "b"], model="qwen-3-4b", stay_attached=False)
    assert list(c.get_job_results(jid2, unpack_json=False).columns) == ["inference_result"]


def test_progress_records_have_the_reference_stream_shape():     # sutro/sdk.py:331-358
    seen = []
    c = Sutro(verbose=False, cache_dir=CACHE, on_progress=seen.append)

    class E:
        def generate(self, rows, progress=None, **kw):
            progress(1, 40, 0)
            progress(1, 30, 5)          # a stale input-token count must not move the state back
            progress(len(rows), 80, 12)
            return GenerationResult([f"o{i}" for i in range(len(rows))], None, None,
                                    {"input_tokens": 80, "output_tokens": 12})
    c.register_engine("qwen-3-4b", E())
    jid = c.infer(["a", "b"], model="qwen-3-4b", stay_attached=False)
    kinds = [r["update_type"] for r in seen]
    assert kinds == ["progress", "tokens"] * 3
    assert [r["result"] for r in seen if r["update_type"] == "progress"] == [1, 1, 2]
    last = seen[-1]["result"]
    assert set(last) == {"input_tokens", "output_tokens", "total_tokens_processed_per_second"}
    assert (last["input_tokens"], last["output_tokens"]) == (80, 12)
    st = c._job(jid).progress
    assert st["rows_done"] == 2 and st["input_tokens"] == 80 and st["output_tokens"] == 12


def test_multi_gpu_engine_merges_shard_progress_and_scatters_rows():
    """MultiGpuEngine host logic with stub shards (no GPU): balanced assignment, job-wide
    row ids, summed progress, positional scatter."""
    from sutro_b200.engine import MultiGpuEngine

    class Shard:
        spec = vocab = tokenizer = None

        def __init__(self, tag):
            self.tag, self.got = tag, None

        def generate(self, rows, row_ids=None, progress=None, **kw):
            self.got = (list(rows), list(row_ids))
            if progress:
                progress(len(rows), 10 * len(rows), len(rows))
            return GenerationResult([f"{r}@{self.tag}" for r in rows], [[i] for i in row_ids],
                                    None, {"n_rows": len(rows), "output_tokens": len(rows)})
    a, b = Shard("a"), Shard("b")
    rows = ["x" * n for n in (9, 1, 5, 7, 3, 2)]
    calls = []
    res = MultiGpuEngine([a, b]).generate(rows, progress=lambda *t: calls.append(t))
    assert [o.split("@")[0] for o in res.outputs] == rows                 # positional
    assert res.out_tokens == [[i] for i in range(6)]                      # job-wide row ids
    assert sorted(a.got[1] + b.got[1]) == list(range(6)) and len(a.got[1]) == len(b.got[1]) == 3
    assert abs(sum(map(len, a.got[0])) - sum(map(len, b.got[0]))) <= 9
    assert calls[-1] == (6, 60, 6) and res.stats["n_rows"] == 6
    blocks = MultiGpuEngine([a, b]).generate(rows, balance="rows")
    assert a.got[1] == [0, 1, 2] and b.got[1] == [3, 4, 5] and blocks.outputs[3] == "xxxxxxx@b"
    with pytest.raises(ValueError):
        MultiGpuEngine([a, b]).generate(rows, balance="tokens")


def test_start_up_calls_of_reference_scripts_are_accepted():
    """`so.set_api_key(...)`, `so.set_base_url(...)`, `so.get_quotas()`, `so.attach(id)` exist
    (sutro/sdk.py:58-95, :759, :1477); dataset calls say where datasets live."""
    c = client()
    c.set_api_key("sk-test")
    c.set_base_url("https://example.invalid")
    c.set_serving_base_url("https://example.invalid")
    assert c.try_authentication("sk-test")["authenticated"] is True
    assert {q["job_priority"] for q in c.get_quotas()} == {0, 1}
    jid = c.infer(["a"], model="qwen-3-4b", stay_attached=False)
    assert c.attach(jid) == interfaces.JobStatus.SUCCEEDED
    with pytest.raises(NotImplementedError):
        c.create_dataset()
    with pytest.raises(NotImplementedError):
        c.upload_to_dataset("d", ["f.parquet"])
    for name in ("set_api_key", "set_base_url", "get_quotas", "attach", "rank", "elo", "infer"):
        assert callable(getattr(so, name))


# --------------------------------------------------------------------------- round-2 fixes
class _CutEngine(StubEngine):
    """One row comes back cut mid-object (what max_tokens below the schema's need does)."""

    def generate(self, rows, **kw):
        r = super().generate(rows, **kw)
        r.outputs[1] = '{"sentiment":"s'
        return r


def test_one_unparsable_row_does_not_disable_json_unpacking():
    c = Sutro(verbose=False, cache_dir=CACHE)
    c.register_engine("qwen-3-4b", _CutEngine())
    job = c.infer(["a", "b", "c"], model="qwen-3-4b", output_schema=Sentiment, stay_attached=False)
    df = c.get_job_results(job)
    got = list(df["sentiment"])
    assert got[0] == "s0" and got[2] == "s2" and pd.isna(got[1])     # pandas shows None as NaN


def test_default_output_budget_comes_from_the_schema():
    """No max_tokens in sampling_params: a schema job gets the longest string its automaton
    accepts (so a constrained row can always finish), free text gets 512."""
    from sutro_b200.schema_fsm import compile_schema

    class Eng(StubEngine):
        class spec:
            max_position = 4096

        def compile_schema(self, schema, limits=None):
            return compile_schema(schema, limits)
    c = Sutro(verbose=False, cache_dir=CACHE)
    eng = Eng()
    c.register_engine("qwen-3-4b", eng)
    enum_schema = {"type": "object", "properties": {"sentiment": {"type": "string", "enum": [
        "positive", "neutral", "negative"]}}, "required": ["sentiment"]}
    c.infer(["x"], model="qwen-3-4b", output_schema=enum_schema, stay_attached=False)
    assert eng.calls[-1][1]["max_new_tokens"] == len('{"sentiment":"positive"}')
    c.infer(["x"], model="qwen-3-4b", stay_attached=False)
    assert eng.calls[-1][1]["max_new_tokens"] == 512
    c.infer(["x"], model="qwen-3-4b", sampling_params={"max_tokens": 7}, stay_attached=False)
    assert eng.calls[-1][1]["max_new_tokens"] == 7


def test_reference_default_model_maps_to_the_local_flagship():
    c = client()
    job = c.infer(["x"], stay_attached=False)            # model defaults to gemma-3-12b-it
    assert c.fetch_job(job)["model"] == "qwen-3-4b"
    with pytest.raises(ValueError, match="Unknown model"):
        c.infer(["x"], model="no-such-model")
    assert not any(j["model"] == "no-such-model" for j in c.list_jobs())   # no FAILED record


def test_files_and_frame_columns_travel_as_arrow(tmp_path):
    """csv / parquet paths and DataFrame columns reach an Arrow-aware engine as ONE Arrow
    column (no Python object per row); lists and multi-column concatenations keep the
    reference's list path (sutro/common.py:111-149)."""
    import pyarrow as pa

    class ArrowEngine(StubEngine):
        def infer_one_call(self, rows, **kw):
            self.calls.append((rows, kw))
            n = len(rows)
            return GenerationResult([f"o{i}" for i in range(n)], None, None,
                                    {"input_tokens": 1, "output_tokens": 1})
    c = Sutro(verbose=False, cache_dir=CACHE)
    eng = ArrowEngine(as_json=False)
    c.register_engine("qwen-3-4b", eng)
    df = pd.DataFrame({"t": ["a", None, "c"], "n": [1, 2, 3]})
    df.to_parquet(tmp_path / "f.parquet")
    df.to_csv(tmp_path / "f.csv", index=False)
    for data in (df, str(tmp_path / "f.parquet"), str(tmp_path / "f.csv")):
        job = c.infer(data, model="qwen-3-4b", column="t", stay_attached=False)
        rows = eng.calls[-1][0]
        assert isinstance(rows, (pa.Array, pa.ChunkedArray)) and len(rows) == 3
        data_b, off = rows_to_blob(rows)
        assert blob_to_rows(data_b, off)[0] == "a" and blob_to_rows(data_b, off)[2] == "c"
        res = c.get_job_results(job, include_inputs=True)
        assert list(res["inputs"])[0] == "a" and len(res) == 3
    c.infer(df, model="qwen-3-4b", column="n", stay_attached=False)       # numbers: their text form
    assert blob_to_rows(*rows_to_blob(eng.calls[-1][0])) == ["1", "2", "3"]
    c.infer(["x", "y"], model="qwen-3-4b", stay_attached=False)
    assert eng.calls[-1][0] == ["x", "y"]
    c.infer(df, model="qwen-3-4b", column=["t", ": ", "n"], stay_attached=False)
    assert eng.calls[-1][0] == ["a: 1", ": 2", "c: 3"]
    with pytest.raises(ValueError, match="Column name must be specified"):
        c.infer(str(tmp_path / "f.parquet"), model="qwen-3-4b")


def test_thinking_models_report_content_and_reasoning():
    """"<model>-thinking" (sutro/common.py:28-32): outputs are {"content", "reasoning_content"}
    objects and get_job_results fans the content's keys out (sutro/sdk.py:1155-1164)."""
    class ThinkEngine(StubEngine):
        class spec:
            max_position = 4096
            embedding_model = False

        def generate(self, rows, **kw):
            self.calls.append((list(rows), kw))
            outs = [f"row {i} looks fine\n</think>\n\n" + json.dumps({"sentiment": f"s{i}"})
                    for i in range(len(rows))]
            return GenerationResult(outs, None, None, {"input_tokens": 1, "output_tokens": 1})
    c = Sutro(verbose=False, cache_dir=CACHE)
    eng = ThinkEngine()
    c.register_engine("qwen-3-4b", eng)
    job = c.infer(["a", "b"], model="qwen-3-4b-thinking", output_schema=Sentiment,
                  sampling_params={"max_thinking_chars": 40, "max_tokens": 99}, stay_attached=False)
    assert eng.calls[-1][1]["thinking_chars"] == 40
    raw = c.get_job_results(job, unpack_json=False)["inference_result"]
    assert json.loads(raw[0]) == {"content": {"sentiment": "s0"}, "reasoning_content": "row 0 looks fine"}
    df = c.get_job_results(job)
    assert list(df["sentiment"]) == ["s0", "s1"] and list(df["reasoning_content"])[1] == "row 1 looks fine"
    # a non-thinking model name does not ask for a thinking turn
    c.infer(["a"], model="qwen-3-4b", output_schema=Sentiment, stay_attached=False)
    assert "thinking_chars" not in eng.calls[-1][1]


def test_client_fsm_limits_reach_the_engine_and_the_output_budget():
    """Strings a schema leaves unbounded stop at FsmLimits.max_string_chars (64 by default; the
    hosted service has no such cap) — the client option raises it, and the default output
    budget follows the longer automaton."""
    from sutro_b200.schema_fsm import FsmLimits, compile_schema
    from sutro_b200.sdk import Sutro

    schema = {"type": "object", "properties": {"note": {"type": "string"}}, "required": ["note"]}
    seen = {}

    class Eng:
        spec = None

        def compile_schema(self, sch, limits=None, thinking_chars=None):
            seen.setdefault("compile", []).append(limits)
            return compile_schema(sch, limits)

        def generate(self, rows, **kw):
            import types
            seen["kw"] = kw
            return types.SimpleNamespace(outputs=['{"note":"x"}'] * len(rows), embeddings=None,
                                         stats={}, cum_logprobs=None)

    wide = FsmLimits(max_string_chars=300)
    c = Sutro(verbose=False, fsm_limits=wide)
    c.register_engine("qwen-3-4b", Eng())
    jid = c.infer(["a", "b"], model="qwen-3-4b", output_schema=schema, stay_attached=False)
    assert jid is not None and seen["kw"]["fsm_limits"] is wide and seen["compile"][-1] is wide
    narrow_budget = compile_schema(schema).longest_path()
    assert seen["kw"]["max_new_tokens"] == compile_schema(schema, wide).longest_path() > narrow_budget
