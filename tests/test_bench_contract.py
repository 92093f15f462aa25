"""bench.py contract.  Without a GPU: the reference arm (`--impl reference`) prints exactly ONE JSON line on stdout
with the agreed keys, also when another rank of a torchrun launch calls it (rank != 0 prints nothing and exits 0), and
our own arm refuses to run without a GPU instead of falling back to the CPU.  On a GPU: --dump-outputs writes the
detections of the timed path."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None, timeout=600):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, env=e, timeout=timeout,
                          stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)


def test_reference_arm_prints_one_json_line():
    r = _run(["--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "0"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "images/sec" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_is_silent_on_other_ranks():
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
             env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_are_the_detections_of_the_timed_path(built, tmp_path):
    """--dump-outputs writes the detections of each workload's last timed step (float32, padding zeroed).  They do not
    depend on the number of timed steps (which --steps sets), i.e. not on which of the two pipeline slots ran last, and
    SSD300's equal what detect_batch returns for the same seeded images and weights."""
    import numpy as np
    names = sorted("%s_%s.npy" % (w, k) for w in ("ssd300", "retinanet800")
                   for k in ("scores", "boxes", "class_id", "count"))
    dumps = []
    for steps in (2, 3):  # after 3 + 4n warm-up steps: the last timed step runs on slot 0, then on slot 1
        out = tmp_path / str(steps)
        r = _run(["--gpus", "1", "--steps", str(steps), "--warmup", "0", "--no-cpu-baseline", "--dump-outputs", str(out)])
        assert r.returncode == 0, r.stderr[-3000:]
        assert json.loads(r.stdout)["steps"] == steps
        assert sorted(p.name for p in out.iterdir()) == names
        dumps.append({n: np.load(str(out / n)) for n in names})
    for n in names:
        assert dumps[0][n].dtype == np.float32, n
        np.testing.assert_array_equal(dumps[0][n], dumps[1][n], err_msg=n)
        if n.endswith("_count.npy"):
            assert dumps[0][n].min() > 0, "the bench's thresholds yield detections in every image"
    got = {k: dumps[0]["ssd300_%s.npy" % k] for k in ("scores", "boxes", "class_id", "count")}
    assert got["scores"].shape[0] == 64 and got["boxes"].shape == got["scores"].shape + (4,)
    import SSD300
    import bench
    det = SSD300.SSD300(dict(bench.CFG), None).detect_batch(bench.synthetic_images(bench.BATCH, seed=0))
    valid = np.arange(det.scores.shape[1])[None, :] < det.count[:, None]
    np.testing.assert_array_equal(got["count"], det.count)
    np.testing.assert_array_equal(got["class_id"], np.where(valid, det.class_id, 0))
    np.testing.assert_array_equal(got["scores"], np.where(valid, det.scores, 0))
    np.testing.assert_array_equal(got["boxes"], np.where(valid[..., None], det.boxes, 0))


def test_own_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    r = _run(["--gpus", "1", "--steps", "1", "--warmup", "3", "--no-cpu-baseline"], timeout=300)
    assert r.returncode != 0 and r.stdout.strip() == ""
