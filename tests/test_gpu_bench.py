"""bench.py contract on the GPU: one JSON line with the metric, the end-to-end arm, the roofline and the CPU baseline;
--dump-outputs writes what the timed path computed."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_line_has_the_contract_keys(tmp_path):
    dump = str(tmp_path / "outputs")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "3",
                          "--n-ref", "30000", "--n-query", "30000", "--cpu-seconds", "1", "--no-config5",
                          "--ref-rows-per-gpu", "300000", "--ref-batch", "60000", "--dump-outputs", dump],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"):
        assert key in line, key
    assert line["n_gpus"] == 1 and line["steps"] == 3 and line["warmup"] == 3 and line["higher_is_better"] is True
    assert line["value"] > 0 and line["gpu_launches"] > 0 and "workload" in line["config"]
    e2e = line["e2e"]
    assert e2e["value"] > 0 and e2e["h2d_bytes_per_step"] == 30000 * 50 * 8 and e2e["d2h_bytes_per_step"] > 0
    assert e2e["value"] != line["value"]
    roof = line["roofline"]
    assert roof["bound"] == "tensor" and 0 < roof["frac"] < 1 and roof["unit"] == "TFLOP/s"
    assert abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-9
    cpu = line["cpu_baseline"]
    assert cpu["kind"] == "port" and cpu["cores"] >= 1 and cpu["value"] > 0 and "sample" in cpu
    assert set(("sm_mhz", "sm_max_mhz", "reasons")) <= set(line["clocks"])
    assert line["mod_canberra"]["value"] > 0 and line["rows_exact_fallback_per_step"] == 0
    assert line["mod_canberra"]["roofline"]["bound"] == "alu" and 0 < line["mod_canberra"]["roofline"]["frac"] < 1
    assert 0 < roof["tmem_readout"]["frac"] < 1.05
    rs = line["ref_sharded"]
    assert rs["value"] > 0 and rs["parity"]["idx_equal"] and rs["parity"]["dist_bit_equal"] and rs["parity"]["weights_bit_equal"]
    assert set(("knn_candidates", "knn_rerank", "exchange", "merge", "snn", "scores")) <= set(rs["stage_ms"])
    assert line["score_determinism"]["bit_identical_single_vs_target_sharded_vs_reference_sharded"] is True
    assert line["projection"]["config1"]["mma"]["ms"] > 0 and line["projection"]["config5_slice"]["mma"]["fp64_tflops"] > 1
    # --dump-outputs: the last timed step's arrays, whole at this size, equal to the same path run here
    import numpy as np
    import torch
    from nabo_b200 import core, synth
    got = {f[:-4]: np.load(os.path.join(dump, f), allow_pickle=False) for f in os.listdir(dump)}
    assert sorted(got) == ["counts", "dist", "idx", "rows", "scores", "weights"]
    assert np.array_equal(got["rows"], np.arange(30000))
    ref = torch.from_numpy(synth.pc_mixture(30000, 50, seed=1)).cuda()
    tgt = torch.from_numpy(synth.pc_mixture(30000, 50, seed=101)).cuda()
    ref_knn, _ = core.knn(ref, ref, 30, "euclidean", drop_first=True, mode="fast")
    idx, dst = core.knn(tgt, ref, 30, "euclidean", mode="fast")
    cnt, w = core.snn_weights(idx, ref_knn, 30)
    sc = core.scores_finalize(core.score_accumulate(idx, cnt, 30000, 30), 30000)
    for name, x in (("idx", idx), ("dist", dst), ("counts", cnt), ("weights", w), ("scores", sc)):
        assert got[name].dtype in (np.float32, np.float64) and np.array_equal(got[name], x.cpu().numpy()), name
