"""bench.py's reference arm runs without a GPU: check the JSON contract of its single output line. On the GPU:
--dump-outputs writes what the timed path computed, the same on every run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-width", "96", "--cpu-height", "64", "--cpu-workers", "2", "--kind", "rgb"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Mpixels/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 2 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("PnnQuantizer") and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.parametrize("args", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "unused"]])
def test_arguments_it_cannot_honour_are_refused(args, tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=120,
                         cwd=tmp_path)
    assert out.returncode == 2 and out.stdout.strip() == "" and not os.listdir(tmp_path), out.stderr[-2000:]


def _channels(argb):
    """(k,) uint32 ARGB -> (k, 4) float32 A, R, G, B: the layout of bench.py --dump-outputs."""
    argb = np.asarray(argb, dtype=np.uint32)
    return np.stack([(argb >> s) & 255 for s in (24, 16, 8, 0)], axis=1).astype(np.float32)


@pytest.mark.parametrize("total,world", [(5000, 1), (5000, 2), (300, 1)])
def test_dump_outputs_layout_and_sample(tmp_path, monkeypatch, total, world):
    """dump_outputs on a CPU tensor whose pixel at flat position p encodes p in its R, G, B channels: the whole output when it
    fits, otherwise DUMP_PIXELS // world distinct sorted positions, the same ones on every call, and each row the pixel there."""
    import types
    import torch
    import bench
    monkeypatch.setattr(bench, "DUMP_PIXELS", 1000)
    pos = np.arange(total, dtype=np.uint32)
    dout = torch.from_numpy((pos | np.uint32(0xFF000000)).view(np.int32))
    dumps = []
    for run in ("a", "b"):
        bench.dump_outputs(types.SimpleNamespace(dump_outputs=str(tmp_path / run)), dout, world - 1, world)
        name = "output_argb.npy" if world == 1 else f"output_argb_rank{world - 1}.npy"
        assert os.listdir(tmp_path / run) == [name]
        dumps.append(np.load(tmp_path / run / name))
    d = dumps[0]
    assert d.dtype == np.float32 and d.shape[1] == 4 and np.array_equal(d, dumps[1])
    assert np.all(d[:, 0] == 255)
    got = (d[:, 1].astype(np.int64) << 16) | (d[:, 2].astype(np.int64) << 8) | d[:, 3].astype(np.int64)
    if total <= 1000 // world:
        assert np.array_equal(got, pos)
    else:
        assert len(got) == 1000 // world and np.all(np.diff(got) > 0) and got[0] >= 0 and got[-1] < total
    assert np.array_equal(d, _channels(got.astype(np.uint32) | np.uint32(0xFF000000)))


@pytest.mark.gpu
def test_dump_outputs_is_what_the_timed_path_computed(tmp_path, oracle):
    from nquant_android_b200 import _build
    from nquant_android_b200.synth import make_image
    _build.build()             # bench.py loads the library as it is: it must be current
    w, h, n = 96, 64, 3
    dumps = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--batch", str(n),
                              "--width", str(w), "--height", str(h), "--no-e2e", "--no-cpu", "--dump-outputs", str(tmp_path / run)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert os.listdir(tmp_path / run) == ["output_argb.npy"]
        dumps.append(np.load(tmp_path / run / "output_argb.npy"))
    assert dumps[0].dtype == np.float32 and dumps[0].shape == (n * w * h, 4)
    assert np.array_equal(dumps[0], dumps[1])
    for i in range(n):         # bench.py's batch: image i from seed 0x5EED0000 + i, converted with seed 0xC0FFEE + i
        ref = oracle.convert(1, make_image(w, h, "noisy", "opaque", seed=0x5EED0000 + i), w, h, 256, True, seed=0xC0FFEE + i, trace=False)
        assert np.array_equal(dumps[0][i * w * h:(i + 1) * w * h], _channels(ref.out)), i
