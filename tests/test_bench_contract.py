"""The one JSON line of bench.py, checked on the arm that runs without a GPU (--impl reference: the CPU restatement on the host cores) and a
2 MB workload: every key of the contract is there, exactly one line is written to stdout, and the workload description (`config`) is what
the GPU arm builds from the same function."""
import importlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--workload", "tiny",
                        "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
                "cpu_baseline", "e2e", "gpu_launches", "schedule"):
        assert key in d, key
    assert d["unit"] == "MB/s" and d["higher_is_better"] is True and d["dtype"] == "u8" and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] == 1 and d["gpu_launches"] == 0
    assert set(("value", "unit", "cores", "kind", "sample")) <= set(d["cpu_baseline"]) and d["cpu_baseline"]["kind"] in ("port", "reference")
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert set(d["levels"]) == {"l3", "l5"} and all(v["compressed_bytes"] > 0 for v in d["levels"].values())
    # the same description object as the GPU arm's (bench.static_config is the only builder of `config`)
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert src.count('"config": static_config(args.workload, passes, BLOCK, NBLOCKS, n, world)') == 2  # reference arm and b200 arm
    assert "workload" in d["config"] and d["config"]["block_size"] == 256 << 10 and d["config"]["uncompressed_bytes"] == 2_000_000
    # --dump-outputs: what the last step computed, whole at this size (the stream of each level and the bytes decoded from it)
    assert sum(f.stat().st_size for f in tmp_path.iterdir()) <= 64 << 20
    synth = importlib.import_module("kanzi-go_b200.synth")
    x = synth.silesia_shaped(2_000_000, seed=synth.SEED + 1)
    for lv in ("l3", "l5"):
        sizes, comp, dec = (np.load(tmp_path / ("%s_%s.npy" % (lv, k))) for k in ("sizes", "compressed", "decompressed"))
        assert sizes.dtype == np.float64 and comp.dtype == np.float32 and dec.dtype == np.float32
        assert list(sizes) == [d["levels"][lv]["compressed_bytes"], 2_000_000] and len(comp) == sizes[0]
        assert np.array_equal(dec, x.astype(np.float32))
