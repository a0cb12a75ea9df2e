"""bench.py contract, CPU side: the reference arm prints exactly ONE JSON line on stdout with the agreed keys (the GPU arm
shares the emit path and the key set is checked on its committed output in profiles/)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
        "data", "config", "e2e"}


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and KEYS <= set(d) and {"cores", "kind", "sample", "value"} <= set(d["cpu_baseline"])
    assert d["cpu_baseline"]["kind"] == "port", d["cpu_baseline"]
    assert d["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] == 0


def test_reference_arm_modules_are_unmodified_and_agree_with_the_port():
    """The reference's TrainModule.forward around its own unmodified STFT / Norm / SpatialNet (wave -> wave on a crop of
    bench.synth_batch, stored by tests/golden/make_golden_parity.py) computes what the op-set port that the CPU arm times
    computes."""
    import numpy as np
    import torch

    sys.path.insert(0, ROOT)
    import bench
    from oracle import eager_gpu as E
    from oracle import spatialnet_oracle as O

    z = np.load(os.path.join(ROOT, "tests", "golden", "train_forward_l2.npz"))
    x = bench.synth_batch(1, 5)[0][..., :128 * 20].contiguous()
    assert abs(x.double().sum().item() - float(z["x_sum"])) < 1e-5, "bench.synth_batch no longer gives the stored input"
    cfg = dict(O.SMALL_CFG, num_layers=2)
    with torch.no_grad():
        est_port = E.io_forward(O.synth_params(cfg, 2), x, cfg, 256, 128, 0)
    assert O.rel_l2(torch.from_numpy(z["est"]), est_port) < 1e-5


def test_committed_gpu_bench_line_has_the_contract_keys():
    d = json.load(open(os.path.join(ROOT, "profiles", "r01_bench_final_b32.json")))
    assert KEYS | {"gpu_launches", "roofline", "cpu_baseline", "clocks"} <= set(d)
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(d["roofline"])
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"]) and d["e2e"]["h2d_bytes_per_step"] > 0
    assert d["config"]["workload"].startswith("SpatialNet-small 6ch F=129 T=250") and d["n_gpus"] == 1
