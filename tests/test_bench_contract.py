"""bench.py contract pieces that need no GPU: the reference arm's JSON line on the small workload (run for real on the host cores: the unmodified
reference from oracle/_ref where it was installed, else the oracle port), rank != 0 of a multi-rank reference launch doing nothing, the workload
tables, and the parser of the committed ncu summary behind roofline.traffic."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None, timeout=900):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=timeout, env=e, cwd=ROOT)


def test_reference_arm_line_small_workload():
    r = _run(["--impl", "reference", "--workload", "conformer_4l256_joint_8x5s", "--steps", "2", "--warmup", "1"])
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["impl"] == "reference" and line["unit"] == "utterances/s" and line["higher_is_better"] is True and line["value"] > 0
    assert line["steps"] == 2 and line["config"]["workload"] == "conformer_4l256_joint_8x5s" and line["gpu_launches"] == 0
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"] and "sample" in cb
    assert line["e2e"] == {"value": line["value"], "unit": "utterances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_without_work():
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"], env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}, timeout=120)
    assert r.returncode == 0 and not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]


def test_workload_tables_and_ncu_summary_parser(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench

    assert set(bench.LM_FUSION) <= set(bench.WORKLOADS) and not (set(bench.STREAMING) & set(bench.WORKLOADS))
    for name, (cfg, secs, batch, beam, ctcw, mlr) in bench.WORKLOADS.items():
        assert cfg["d_model"] % cfg["heads"] == 0 and secs > 0 and batch > 0 and 0 < beam <= 64 and 0.0 <= ctcw <= 1.0 and mlr < 0, name
    prof = tmp_path / "profiles"
    prof.mkdir()
    (prof / "r02_ncu_gemm_2cta_ffn_w1_ew16_summary.txt").write_text(
        "== kernel\n   gpu__time_duration.sum      500.5 us\n   dram__bytes_read.sum   1.5 Gbyte\n   dram__bytes_write.sum   250 Mbyte\n"
        "   sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active    77.7 %\n")
    monkeypatch.setattr(bench, "ROOT", str(tmp_path))
    monkeypatch.setattr(bench, "NCU_TRAFFIC", dict(bench.NCU_TRAFFIC))
    bench._load_ncu_traffic()
    t = bench.NCU_TRAFFIC
    assert abs(t["dram_bytes"] - 1.75e9) < 1 and t["gpu_time_us_under_ncu"] == 500.5 and t["tensor_pipe_active_pct"] == 77.7 and "r02" in t["source"]


def test_dump_outputs_layout(tmp_path):
    """--dump-outputs: the top `nbest` hypotheses per utterance as float64 arrays, padded with -1 (tokens) / NaN (scores)."""
    import numpy as np
    import torch

    sys.path.insert(0, ROOT)
    import bench
    from espnet_b200.search import Hypothesis

    res = [[Hypothesis(yseq=torch.tensor([9, 3, 4, 9]), score=-1.5, scores={"decoder": -1.0, "ctc": -2.5}),
            Hypothesis(yseq=torch.tensor([9, 9]), score=-3.0, scores={"decoder": -2.0, "ctc": -5.0}),
            Hypothesis(yseq=torch.tensor([9, 5, 9]), score=-4.0, scores={"decoder": -3.0, "ctc": -7.0})], []]
    names = bench.dump_outputs(str(tmp_path / "out"), res, 2)
    assert names == ["hyp_score", "hyp_score_ctc", "hyp_score_decoder", "hyp_yseq"]
    a = {n: np.load(tmp_path / "out" / f"{n}.npy") for n in names}
    assert all(v.dtype == np.float64 for v in a.values())
    np.testing.assert_array_equal(a["hyp_yseq"], [[[9, 3, 4, 9], [9, 9, -1, -1]], [[-1] * 4] * 2])
    np.testing.assert_array_equal(a["hyp_score"], [[-1.5, -3.0], [np.nan, np.nan]])
    np.testing.assert_array_equal(a["hyp_score_ctc"], [[-2.5, -5.0], [np.nan, np.nan]])
