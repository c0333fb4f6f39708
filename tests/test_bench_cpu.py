"""bench.py is the file the driver runs unattended: check on CPU that it imports, parses its
command line, and that its host-only helpers work (the GPU arms need a B200)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_imports_and_prints_usage():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--rows", "--workload",
                 "--no-secondary", "--dump-outputs"):
        assert flag in out.stdout


def test_dump_outputs_round_trip_and_sample(tmp_path):
    sys.path.insert(0, ROOT)
    import numpy as np
    import bench
    from sutro_b200 import vocab as VB
    outs = ['{"sentiment":"positive"}', '{"sentiment":"neutral"}', "café 🙂 \ufffd", ""] * 50

    def read(d):
        a, idx = np.load(d / "inference_result.npy"), np.load(d / "row_index.npy")
        assert a.dtype == np.float32 and idx.dtype == np.float64
        rows = ["".join(chr(int(x)) for x in r if x >= 0) for r in a]
        return a.shape, rows, idx.astype(int).tolist()

    bench.dump_outputs(str(tmp_path / "all"), outs, width=30)
    shape, rows, idx = read(tmp_path / "all")
    assert shape == (len(outs), 30) and rows == outs and idx == list(range(len(outs)))
    # over the limit: a seeded sample whose rows and shape depend on the row count and the
    # width only, not on what the rows hold; the files stay within the limit
    limit = 4096 + 40 * (4 * 30 + 8)
    bench.dump_outputs(str(tmp_path / "s1"), outs, width=30, limit=limit)
    bench.dump_outputs(str(tmp_path / "s2"), ["x"] * len(outs), width=30, limit=limit)
    for d in ("s1", "s2"):
        assert sum(f.stat().st_size for f in (tmp_path / d).iterdir()) <= limit
    shape, rows, idx = read(tmp_path / "s1")
    assert shape == (40, 30) and idx == sorted(idx) and rows == [outs[i] for i in idx]
    assert read(tmp_path / "s2")[::2] == (shape, idx)
    # the width bounds every result the job can return: max_new_tokens tokens of the vocabulary
    v = VB.build_vocab("qwen3", 1024, seed=0)
    assert bench.dump_width(v, 24) == 24 * max(len(b) for b in v.token_bytes)


def test_host_helpers():
    sys.path.insert(0, ROOT)
    import bench
    from sutro_b200 import synth
    rows = synth.product_reviews(500, seed=0)
    p = bench.plumbing_cost("qwen-3-4b", rows, ['{"sentiment":"positive"}'] * len(rows))
    assert p["rows"] == 500 and p["rows_per_s"] > 0 and p["payload_bytes"] > 500
    t = bench.ncu_traffic("r02_ncu_prefill_step.csv", "gemm2_bf16_tn_kernel<2, 7")
    assert t is not None and 0.9e9 < t < 2.5e9       # one gate/up launch: ~0.9 GB algorithmic
    t = bench.ncu_traffic("r02_ncu_decode_side.csv", "attn_decode_warp_kernel")
    assert t is not None and t > 1e8
    assert bench.ncu_traffic("does_not_exist.csv", "x") is None
    pk = bench.peaks()
    assert pk["hbm_gbs"] > 1000 and pk["bf16_tflops_sustained"] > 100
    json.dumps(bench.SCHEMA)
    assert len(bench.make_rows(7, seed=1)) == 7
    # the nested configs[4] schema compiles, and the frame shape SURVEY.md §8d names is met:
    # synthetic reviews average ~96 tokens under the synthetic vocabulary
    from sutro_b200.schema_fsm import FsmLimits, compile_schema
    d = compile_schema(bench.ORDER_SCHEMA, FsmLimits(max_string_chars=12, max_array_items=3))
    assert d.matches(b'{"customer":"x","items":[{"name":"a","quantity":3,"kind":"b","price":null}],'
                     b'"paid":true}')
    kw = bench.infer_kwargs("qwen-3-4b")
    assert kw["output_schema"] == bench.SCHEMA and kw["column"] == bench.COLUMN


def test_synthetic_review_length_matches_the_survey_shape():
    sys.path.insert(0, ROOT)
    import numpy as np
    from oracle.bpe_ref import RefTokenizer
    from sutro_b200 import modelspec as MS
    from sutro_b200 import synth, vocab as VB
    spec = MS.get_spec("qwen-3-4b")
    tok = RefTokenizer(VB.build_vocab(spec.family, spec.vocab_size, seed=0))
    n = [len(tok.encode(r)) for r in synth.product_reviews(400, seed=5)]
    assert 80 <= np.mean(n) <= 110 and min(n) >= 12 and max(n) <= 300, (np.mean(n), min(n), max(n))
    assert tok.decode(tok.encode("round trip, 100% exact")) == "round trip, 100% exact"


def test_smoke_and_build_entry_points_exist():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as g
    assert callable(g.build) and callable(g.smoke)
