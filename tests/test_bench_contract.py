"""CPU: the reference arm of bench.py (`--impl reference`) runs without a GPU and prints the JSON line the driver reads.
The arm times the CPU oracle port of the path (the one other place bench.py may execute oracle/), so this also checks that
the line names the same workload / metric / unit as the GPU arm's config table."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference"
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in line, k
    assert line["unit"] == "Gsamples/s" and line["higher_is_better"] is True and line["value"] > 0
    assert line["steps"] == 1 and line["n_gpus"] == 1 and line["gpu_launches"] == 0
    assert line["config"]["workload"] == "c2_fft1024_u8iq_2p28"          # BASELINE.json configs[1], the headline
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    e = line["e2e"]
    assert e["value"] == line["value"] and e["unit"] == line["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0

    # the GPU arm describes the same workload with the same config object
    sys.path.insert(0, ROOT)
    import bench
    assert bench.config_dict("c2") == line["config"]


def test_dump_outputs_format_and_row_sample(tmp_path, monkeypatch):
    """--dump-outputs: float32 files, complex values with a trailing (re, im) axis, flags as 0 / 1; an output over its
    share of the budget is written as the seeded sample of its rows (a 1-D stream cut into blocks of DUMP_ROW samples),
    the same rows on every call; the files together stay within the budget."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    monkeypatch.setattr(bench, "DUMP_ROW", 256)
    g = torch.Generator().manual_seed(1)
    outs = {"stream": torch.randn(100000, dtype=torch.complex64, generator=g),
            "flags": torch.randint(0, 2, (64, 4096), dtype=torch.uint8, generator=g),
            "small": torch.randn(10, 3, generator=g)}
    bench.dump_outputs(torch, outs, str(tmp_path / "a"))
    bench.dump_outputs(torch, outs, str(tmp_path / "b"))
    share = (1 << 20) // 3
    rows = bench.sample_rows(100000 // 256, share // (256 * 8))
    want = {"stream": torch.view_as_real(outs["stream"][:100000 // 256 * 256].view(-1, 256)).numpy()[rows],
            "flags": outs["flags"].float().numpy()[bench.sample_rows(64, share // (4096 * 4))],
            "small": outs["small"].numpy()}
    total = 0
    for name, w in want.items():
        a, b = np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy"))
        assert a.dtype == np.float32 and np.array_equal(a, w) and np.array_equal(a, b), name
        total += os.path.getsize(tmp_path / "a" / (name + ".npy"))
    assert len(rows) > 100 and total <= (1 << 20) + 3 * 128


@pytest.mark.gpu
def test_gpu_arm_steps_and_reproducible_dump(tmp_path):
    """--steps K times K steps (the library's launches in the timed region scale with K), and --dump-outputs writes the
    same files on every run with the same arguments (the stateless FFT for any K; the decimating FIR, whose history and
    phase carry between steps, for equal K), under 64 MB, holding what the path computes (rows checked with the oracle)."""
    import numpy as np
    import torch
    import oracle_lib as O
    sys.path.insert(0, ROOT)
    import bench

    def run(tag, *extra):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--no-cpu", "--no-e2e", "--configs", "none",
                            "--dump-outputs", str(tmp_path / tag)] + list(extra),
                           capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert p.returncode == 0, p.stderr[-2000:]
        files = sorted(os.listdir(tmp_path / tag))
        assert sum(os.path.getsize(tmp_path / tag / f) for f in files) <= 64_000_000
        return json.loads(p.stdout.strip().splitlines()[-1]), {f: np.load(tmp_path / tag / f) for f in files}

    a, da = run("a", "--workload", "c2_small", "--steps", "2")
    b, db = run("b", "--workload", "c2_small", "--steps", "6")
    assert (a["steps"], b["steps"]) == (2, 6) and a["gpu_launches"] > 0 and b["gpu_launches"] == 3 * a["gpu_launches"]
    assert list(da) == ["spectrum.npy"] and np.array_equal(da["spectrum.npy"], db["spectrum.npy"])
    spec = da["spectrum.npy"]
    assert spec.dtype == np.float32 and spec.shape[1:] == (1024, 2)
    rows = bench.sample_rows(1 << 14, spec.shape[0])
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(bench.SEED + 2)
    raw = torch.randint(0, 256, (2 << 24,), dtype=torch.uint8, device=dev, generator=gen).cpu().numpy().reshape(-1, 2048)
    for i in (0, len(rows) // 2, len(rows) - 1):
        ref = O.fft_batch_u8(raw[rows[i]], 1024, 1)[0]
        got = spec[i, :, 0] + 1j * spec[i, :, 1]
        assert np.abs(got - ref).max() / np.abs(ref).max() < 1e-4, i

    _, fa = run("c", "--workload", "c3", "--steps", "3")
    _, fb = run("d", "--workload", "c3", "--steps", "3")
    assert list(fa) == ["filtered.npy"] and fa["filtered.npy"].shape[1] == 2
    assert abs(fa["filtered.npy"].shape[0] - (1 << 26) / 10) <= 1
    assert np.array_equal(fa["filtered.npy"], fb["filtered.npy"])
