"""bench.py's reference arm (`--impl reference`) on a tiny workload, on the CPU: one JSON line with the keys its readers
rely on, no product library mapped into the process (the arm times the CPU restatement of the reference alone), the
silent exit of ranks other than 0 under torchrun, and the outputs --dump-outputs writes."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra=None, extra_args=()):
    env = dict(os.environ)
    env.update(env_extra or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--channels", "8", "--seconds", "0.25", "--steps", "2",
                           "--warmup", "1", *extra_args], capture_output=True, text=True, cwd=ROOT, env=env, timeout=300)


def test_reference_arm_prints_one_contract_line():
    r = _run()
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] == "GC-ADPCM encode Msamples/sec (batch)" and line["unit"] == "Msamples/s"
    assert line["higher_is_better"] is True and line["steps"] == 2 and line["warmup"] == 1 and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"]


def test_reference_arm_other_ranks_exit_silently():
    r = _run({"RANK": "3", "LOCAL_RANK": "3", "WORLD_SIZE": "8"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_reference_arm_does_not_map_the_product_library():
    code = ("import sys, runpy\n"
            "sys.argv = ['bench.py', '--impl', 'reference', '--channels', '4', '--seconds', '0.1', '--steps', '1', '--warmup', '0']\n"
            "try:\n    runpy.run_path('bench.py', run_name='__main__')\nexcept SystemExit:\n    pass\n"
            "maps = open('/proc/self/maps').read()\n"
            "print('MAPPED' if 'libvgaudio_b200' in maps else 'CLEAN')\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, timeout=300)
    assert r.returncode == 0, r.stderr
    assert r.stdout.strip().endswith("CLEAN")


def test_reference_arm_dumps_the_last_step(tmp_path, oracle):
    spec = importlib.util.spec_from_file_location("vgb_synth", os.path.join(ROOT, "vgaudio_b200", "synth.py"))
    synth = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(synth)
    dumps = []
    for run in ("a", "b"):
        r = _run(extra_args=("--dump-outputs", str(tmp_path / run)))
        assert r.returncode == 0, r.stderr
        dumps.append({name: np.load(tmp_path / run / f"{name}.npy") for name in ("coefs", "adpcm")})
    pcm = np.stack([synth.channel(4 + i, 12000) for i in range(8)])
    coefs, adpcm, _ = oracle.encode_batch(pcm)
    for d in dumps:
        assert d["coefs"].dtype == np.float32 and d["adpcm"].dtype == np.float32
        assert np.array_equal(d["coefs"], coefs) and np.array_equal(d["adpcm"], adpcm)


def test_dump_sample_stays_within_budget():
    import bench

    for n_ch, n_bytes in ((1024, 822858), (3, 40_000_000), (8, 6858)):
        rows, width = bench.dump_sample(n_ch, n_bytes)
        assert 4 * len(rows) * (16 + width) <= bench.DUMP_BYTES
        assert len(rows) >= 1 and np.all(np.diff(rows) > 0) and rows[0] >= 0 and rows[-1] < n_ch
        assert np.array_equal(rows, bench.dump_sample(n_ch, n_bytes)[0])
    assert bench.dump_sample(8, 6858)[1] == 6858 and len(bench.dump_sample(8, 6858)[0]) == 8


@pytest.mark.gpu
def test_device_path_dumps_the_last_step(tmp_path, oracle):
    import torch

    import bench

    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--channels", "8", "--seconds", "0.25", "--steps", "2",
                        "--warmup", "1", "--no-e2e", "--no-cpu", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr
    pcm = bench.make_batch_gpu(torch, 8, 12000, 0, torch.device("cuda", 0)).cpu().numpy()
    coefs, adpcm, _ = oracle.encode_batch(pcm)
    assert np.array_equal(np.load(tmp_path / "coefs.npy"), coefs)
    assert np.array_equal(np.load(tmp_path / "adpcm.npy"), adpcm)
