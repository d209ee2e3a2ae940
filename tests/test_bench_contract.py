"""bench.py output contract on a CPU-only box: the reference arm (`--impl reference`, the oracle port of the reference's CPU
path) prints ONE JSON line with the keys the driver reads; the b200 arm refuses to run without a GPU (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(*args, timeout=600):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout, cwd=ROOT)


def test_reference_arm_json_line():
    r = run("--impl", "reference", "--tiny", "--steps", "1", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(line) == 1
    j = json.loads(line[0])
    assert j["impl"] == "reference" and j["unit"] == "crops/s" and j["higher_is_better"] is True and j["n_gpus"] == 1
    assert j["steps"] == 1 and j["warmup"] == 1 and j["value"] > 0 and j["ms_per_step"] > 0
    assert set(j["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"}
    assert j["e2e"]["h2d_bytes_per_step"] == 0 and j["e2e"]["d2h_bytes_per_step"] == 0 and j["e2e"]["value"] == j["value"]
    cb = j["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == j["value"] and isinstance(cb["sample"], str)
    assert "workload" in j["config"]


def test_dump_outputs_writes_what_a_step_returned(tmp_path):
    """bench.dump_outputs on lock-step stub searches (one succeeds at its root with three valid boxes, two walk the tree) and
    stand-in option scorings: finite float32 / float64 arrays holding the step's results, search paths concatenated"""
    import numpy as np

    import bench
    from tests.helpers import NumpyScorer, RecordStub, synth_image
    from vstar_b200.visual_search import visual_search_many
    jobs = [(synth_image(24, 1280, 960), "mug", 224), (synth_image(27, 2000, 420), "mug", 224), (synth_image(28, 1001, 577), "mug", 251)]
    results, states = visual_search_many(RecordStub("root"), jobs, batch_size=8, scorer=NumpyScorer(),
                                         target_cue_threshold=-1e9, target_cue_threshold_minimum=-1e9)
    scored = [(torch.tensor([1.5, 0.25, 2.0, 3.0]) + i, i % 4) for i in range(len(jobs))]
    out = tmp_path / "out"
    bench.dump_outputs(str(out), results, states, scored)
    got = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert all(f.endswith(".npy") for f in os.listdir(out)) and all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert all(np.isfinite(a).all() for a in got.values()), [k for k, a in got.items() if not np.isfinite(a).all()]
    assert got["search_path_length"].tolist() == [pl for _, pl, _, _ in results]
    assert got["search_success"].tolist() == [float(ok) for _, _, ok, _ in results]
    assert np.array_equal(got["search_final_bbox"], [fs["bbox"] for fs, _, _, _ in results])
    assert np.array_equal(got["search_detection_result"], np.stack([fs["detection_result"].numpy() for fs, _, _, _ in results]))
    lengths = [len(st.search_path) for st in states]
    assert lengths[0] == 1 and min(lengths[1:]) > 1 and got["search_path_nodes"].tolist() == lengths
    nodes = [node for st in states for node in st.search_path]
    assert np.array_equal(got["search_path_bbox"], [node["bbox"] for node in nodes])
    assert np.array_equal(got["search_path_score"], [node["score"] or 0.0 for node in nodes])
    roots = np.cumsum([0] + lengths[:-1])
    assert (got["search_path_score"][roots] == 0).all()
    det = [node.get("temp_detection_result") for node in nodes]
    assert got["search_path_detected"].tolist() == [float(d is not None) for d in det] and 0 < sum(d is not None for d in det) < len(det)
    for k, d in enumerate(det):
        want_logit, want_box = (0.0, np.zeros(4)) if d is None else (float(d[0]), d[1].numpy())
        assert got["search_path_top_logit"][k] == want_logit and np.array_equal(got["search_path_box"][k], want_box)
    av = results[0][3]
    assert len(av) == 3 and np.array_equal(got["search_valid_boxes"], av.numpy())
    assert got["search_valid_boxes_count"].tolist() == [3, 0, 0]
    assert got["vqa_option_losses"].dtype == np.float32
    assert np.array_equal(got["vqa_option_losses"], np.stack([losses.numpy() for losses, _ in scored]))
    assert got["vqa_choice"].tolist() == [c for _, c in scored]


def test_dump_outputs_needs_the_b200_arm(tmp_path):
    r = run("--impl", "reference", "--dump-outputs", str(tmp_path / "out"), timeout=120)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not (tmp_path / "out").exists()


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-only check")
def test_b200_arm_needs_a_gpu():
    r = run("--tiny", "--steps", "1", "--warmup", "1", "--no-cpu-baseline", timeout=300)
    assert r.returncode != 0                       # fails loudly: there is no CPU / PyTorch fallback for the product path
    assert "{\"metric\"" not in r.stdout
