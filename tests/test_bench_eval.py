"""V*Bench driver (vstar_b200.bench_eval) against the output of the REFERENCE's own eval_model
(/root/reference/vstar_bench_eval.py:168-273) run on the same tiny synthetic benchmark tree with the same stub VQA / stub VSM
(golden produced by oracle/make_golden.py:case_bench_eval)."""
import json
import os
import types

import pytest

from tests.helpers import NumpyScorer, StubVQA, StubVSM, make_bench_folder

GOLD = os.path.join(os.path.dirname(__file__), "golden", "bench_eval_golden.json")


def run(tmp_path, in_flight, tag):
    from vstar_b200.bench_eval import eval_model
    # the driver takes an annotation's path to be its image's path up to the first '.' (as the reference does), so the
    # tree is named relative to tmp_path (the working directory), whose own path may contain dots
    folder = make_bench_folder("bench")
    out = str(tmp_path / f"out_{tag}.json")
    args = types.SimpleNamespace(benchmark_folder=folder, output_path=out, vsm_model_path="stub", minimum_size_scale=4.0,
                                 minimum_size=224, images_in_flight=in_flight, search_batch=8)
    lines = []
    res, overall = eval_model(args, vqa_llm=StubVQA(), vsm=StubVSM(), log=lambda *a: lines.append(a),
                              search_kwargs=dict(scorer=NumpyScorer()))
    return res, overall, json.load(open(out)), lines


def check_against_golden(res):
    gold = json.load(open(GOLD))
    assert list(res.keys()) == list(gold.keys()) == ["direct_attributes", "relative_position"]
    for t in gold:
        got = {r["image"]: r for r in res[t]}
        assert sorted(got) == [g["image"] for g in gold[t]]
        for g in gold[t]:
            r = got[g["image"]]
            assert list(r.keys()) == list(g.keys())          # same keys in the same order as the reference's JSON
            for k in ("question", "options", "prediction_freeform", "missing_objects", "option_chosen", "correct"):
                assert r[k] == g[k], (g["image"], k)
            assert [s["name"] for s in r["search_result"]] == [s["name"] for s in g["search_result"]]
            for a, b in zip(r["search_result"], g["search_result"]):
                assert a["bbox"] == pytest.approx(b["bbox"], abs=1e-3)


@pytest.mark.parametrize("in_flight", [1, 3, 8])
def test_matches_reference_driver(tmp_path, monkeypatch, in_flight):
    monkeypatch.chdir(tmp_path)
    res, overall, dumped, lines = run(tmp_path, in_flight, str(in_flight))
    assert dumped == json.loads(json.dumps(res))
    check_against_golden(dumped)
    gold = json.load(open(GOLD))
    n = sum(len(v) for v in gold.values())
    assert overall == pytest.approx(sum(g["correct"] for v in gold.values() for g in v) / n)
    assert [l[0] for l in lines[:2]] == ["direct_attributes", "relative_position"] and len(lines) == 3


def test_cli_parser_matches_reference_flags():
    from vstar_b200.bench_eval import build_parser
    a = build_parser().parse_args([])
    # names / defaults of vstar_bench_eval.py:275-284
    assert (a.vqa_model_path, a.vqa_model_base, a.conv_type, a.benchmark_folder, a.vsm_model_path, a.output_path,
            a.minimum_size_scale, a.minimum_size) == ("craigwu/seal_vqa_7b", None, "v1", "vstar_bench", "craigwu/seal_vsm_7b",
                                                      "eval_result.json", 4.0, 224)
