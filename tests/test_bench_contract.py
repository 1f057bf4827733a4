"""bench.py contract on a box without a GPU: the reference arm (the reference's own CPU path, oracle/_ref or the
oracle port) runs anywhere and must print exactly one JSON line with the keys the driver reads; the GPU arm must
refuse to run without a device instead of falling back to anything."""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, str(ROOT / "bench.py")] + args, capture_output=True, text=True, cwd=ROOT,
                          env=e, timeout=600)


@pytest.mark.timeout(600)
def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    from sr_object_detection_b200 import build
    build.build()
    if not ((ROOT / "oracle" / "_ref" / "darknet_ref").exists() or (ROOT / "oracle" / "_build" / "y2_oracle").exists()):
        pytest.skip("oracle binaries not built")
    # torchrun exports OMP_NUM_THREADS=1 to its workers: the arm must set the thread count itself
    r = _run(["--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "0"], env={"OMP_NUM_THREADS": "1"})
    assert r.returncode == 0, r.stderr[-400:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "images/sec" and d["unit"] == "images/s"
    assert d["higher_is_better"] is True and d["steps"] == 1 and d["n_gpus"] == 1 and d["value"] > 0
    assert d["config"]["workload"].startswith("yolo-voc.cfg 416x416 batch 64")
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["cores"] == d["config"]["omp_threads"] == len(os.sched_getaffinity(0))
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_silently():
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"], env={"RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.skipif(torch.cuda.is_available(), reason="needs a box without a GPU")
def test_gpu_arm_fails_loudly_without_a_device():
    r = _run(["--steps", "1", "--warmup", "3"])
    assert r.returncode != 0
    assert r.stdout.strip() == "", "no bench line may be printed without a device"


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_gpu_arm_dumps_the_last_timed_step_identically_run_to_run(tmp_path):
    """--steps sets the timed steps; --dump-outputs writes what network_detect_wait returned after the last one: the
    detections one network_detect_batch computes on the same seeded weights and images, and the same bytes on two
    runs with the same arguments."""
    import bench
    from sr_object_detection_b200 import darknet as dn
    from sr_object_detection_b200 import synth
    batch = 8
    dumps = []
    for k in range(2):
        out = tmp_path / f"run{k}"
        r = _run(["--gpus", "1", "--steps", "2", "--warmup", "3", "--batch", str(batch), "--no-cpu-baseline",
                  "--dump-outputs", str(out)])
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
        files = {p.name: np.load(p) for p in sorted(out.iterdir())}
        assert sorted(files) == ["counts.npy", "detections.npy"]
        assert all(a.dtype in (np.float32, np.float64) for a in files.values())
        dumps.append(files)
    for name in dumps[0]:
        assert dumps[0][name].tobytes() == dumps[1][name].tobytes(), name

    cfg, weights = bench._write_inputs(tmp_path, batch)
    dn.set_gpu_index(0)
    net = dn.parse_network_cfg(cfg)
    dn.load_weights(net, weights)
    images = synth.images(batch, 3, bench.SIDE, bench.SIDE, seed=bench.SEED_X)
    per_image, counts = dn.network_detect_batch(net, images, bench.THRESH, bench.NMS, bench.MAX_DET)
    dn.free_network(net)
    assert all(c > 0 for c in counts), "the bench workload must produce detections"
    want = np.concatenate([np.stack([np.full(len(d), b), d["box_index"], d["obj_id"], d["prob"], d["x"], d["y"], d["w"],
                                     d["h"]], axis=1).astype(np.float64) for b, d in enumerate(per_image)])
    assert dumps[0]["counts.npy"].tolist() == counts
    assert dumps[0]["detections.npy"].shape == want.shape
    assert dumps[0]["detections.npy"].tobytes() == want.tobytes()
