"""CPU tier: the parts of bench.py's contract that need no GPU -- the reference arm (`--impl reference`: the compiled,
unmodified reference timed on the host cores) prints one JSON line with the contract's keys; ranks other than 0 print
nothing; the B200 arm fails loudly without a device instead of falling back."""
import json
import os
import subprocess
import sys

import pytest

from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(not O.have_ref(), reason="oracle/_ref not built")
@pytest.mark.parametrize("workload", ["config2_small", "curvature3_small"])
def test_reference_arm_line(workload):
    """(smoke-size workloads: the default one is 512^3 x 5 variables, minutes of host time)"""
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "3", "--workload", workload],
                       capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Gcells/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and d["vs_baseline"] is None and "workload" in d["config"]
    # the reference arm runs the WHOLE workload (same grid, every variable): its config object is the B200 arm's
    import bench
    spec = bench.workload_spec(workload)
    assert d["config"] == bench.config_of(spec, spec["build"](fill=False))
    assert d["steps"] == 2 and d["metric"] == bench.metric_name(spec["kind"])
    # under torchrun only rank 0 runs the reference
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    q = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True, text=True, cwd=ROOT, env=env, timeout=120)
    assert q.returncode == 0 and q.stdout.strip() == ""


def test_dump_outputs_sample(tmp_path, monkeypatch):
    """--dump-outputs: one float64 file per output component, every cell in host-concat order while the budget allows, else
    the same seeded sample of cells in every component and every run, within the budget."""
    import numpy as np
    import bench
    spec = bench.workload_spec("curvature3_small")
    pf = spec["build"](fill=False)

    class H:
        levels = pf.levels
        num_cells = sum(l.ncells for l in pf.levels)

    class Out:                                   # stands for the device Field: cell value = its host-concat index + component
        def download_box(self, l, b, c):
            off = sum(lv.ncells for lv in pf.levels[:l]) + sum(
                int(np.prod([hi[d] - lo[d] + 1 for d in range(3)])) for lo, hi in pf.levels[l].boxes[:b])
            lo, hi = pf.levels[l].boxes[b]
            n = [hi[d] - lo[d] + 1 for d in range(3)]
            return (off + np.arange(n[0] * n[1] * n[2], dtype=np.float64)).reshape(n[2], n[1], n[0]) + 0.25 * c

    names = bench.output_names(spec)
    bench.dump_outputs(spec, H, Out(), str(tmp_path / "all"))
    for c, n in enumerate(names):
        a = np.load(str(tmp_path / "all" / (n + ".npy")))
        assert a.dtype == np.float64 and np.array_equal(a, np.arange(H.num_cells) + 0.25 * c)
    monkeypatch.setattr(bench, "DUMP_BYTES", 8 * len(names) * 1000)
    for run in ("s1", "s2"):
        bench.dump_outputs(spec, H, Out(), str(tmp_path / run))
    idx = np.load(str(tmp_path / "s1" / "Progress.npy"))
    assert idx.size == 1000 and np.all(np.diff(idx) > 0) and idx[-1] < H.num_cells
    for c, n in enumerate(names):
        a, b = np.load(str(tmp_path / "s1" / (n + ".npy"))), np.load(str(tmp_path / "s2" / (n + ".npy")))
        assert np.array_equal(a, b) and np.array_equal(a, idx + 0.25 * c)
    assert sum(f.stat().st_size for f in (tmp_path / "s1").iterdir()) <= 8 * len(names) * 1000 + 128 * len(names)


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["config2_small", "curvature3_small"])
def test_dump_outputs_match_oracle(gpu, tmp_path, workload):
    """bench.py --dump-outputs end to end: the files hold the real Field's outputs in their component order, bit for bit the
    oracle's on the inputs bench.py generates (config2_small is sampled, curvature3_small written whole)."""
    import numpy as np
    import torch
    import bench
    out = tmp_path / "dump"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--steps", "1", "--no-extras",
                        "--no-cpu-baseline", "--e2e-steps", "0", "--dump-outputs", str(out)], capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert p.returncode == 0, p.stderr[-2000:]
    spec = bench.workload_spec(workload)
    names = bench.output_names(spec)
    assert sorted(os.listdir(str(out))) == sorted(n + ".npy" for n in names)
    pf = spec["build"](fill=False)
    idx = bench.dump_cells(sum(l.ncells for l in pf.levels), len(names))
    host = bench.gen_fields(torch, pf.levels, [list(range(len(l.boxes))) for l in pf.levels], spec["names"])
    OH = O.OracleHier(pf)
    for v in range(len(spec["names"])):
        s = np.concatenate([host[l][v].numpy() for l in range(len(pf.levels))])
        want = OH.grad(s) if spec["kind"] == "grad" else OH.curvature(s, float(s.min()), float(s.max()))
        for c in range(len(want)):
            got = np.load(str(out / (names[len(want) * v + c] + ".npy")))
            assert got.dtype == np.float64 and np.array_equal(got, want[c][idx]), (workload, names[len(want) * v + c])


def test_b200_arm_needs_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--no-extras", "--no-cpu-baseline"],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert p.returncode != 0 and not any(l.startswith("{") for l in p.stdout.splitlines())
