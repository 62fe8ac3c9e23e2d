"""CPU: the JSON-line contract of bench.py's reference arm (the CPU oracle port timed on this box's cores) and the
argument surface the driver uses.  The GPU arm needs a device and is exercised on the B200 box."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["steps"] == 1 and d["warmup"] == 0 and d["n_gpus"] == 1 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_writes_float32_and_samples_large_arrays_at_fixed_positions(tmp_path, monkeypatch):
    import numpy as np
    import pytest
    import torch
    import bench
    gen = torch.Generator().manual_seed(0)
    big = torch.randn(40, 50, generator=gen).to(torch.bfloat16)
    small = torch.randn(7, 5, generator=gen)
    arrays = [("loss", torch.tensor(1.5), 16), ("param.big", big, 500), ("grad.small", small, 500)]
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    got = {n: np.load(tmp_path / "a" / (n + ".npy")) for n, _, _ in arrays}
    for n, a in got.items():
        assert a.dtype == np.float32 and np.array_equal(a, np.load(tmp_path / "b" / (n + ".npy"))), n
    assert got["loss"] == 1.5 and np.array_equal(got["grad.small"], small.numpy())
    assert got["param.big"].shape == (500,) and np.isin(got["param.big"], big.float().numpy()).all()
    monkeypatch.setattr(bench, "DUMP_BYTES", 4 * 500)
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "c"), arrays)
    assert not (tmp_path / "c").exists()


def test_reset_training_state_makes_the_next_step_a_first_step():
    import torch
    import bench
    x = torch.randn(8, 6, generator=torch.Generator().manual_seed(1))
    for make_opt in (lambda ps: torch.optim.Adam(ps, lr=1e-2, foreach=False),
                     lambda ps: torch.optim.SGD(ps, lr=1e-2, momentum=0.9, weight_decay=1e-4, foreach=False)):
        torch.manual_seed(0)
        fresh, used = torch.nn.Linear(6, 5), torch.nn.Linear(6, 5)
        used.load_state_dict(fresh.state_dict())
        initial = [p.detach().clone() for p in used.parameters()]
        o_fresh, o_used = make_opt(list(fresh.parameters())), make_opt(list(used.parameters()))

        def step(m, o):
            o.zero_grad()
            (m(x) ** 2).sum().backward()
            o.step()

        for _ in range(3):
            step(used, o_used)
        bench.reset_training_state(list(used.parameters()), initial, o_used)
        assert all(torch.equal(p, q) for p, q in zip(used.parameters(), fresh.parameters()))
        step(fresh, o_fresh)
        step(used, o_used)
        assert all(torch.equal(p, q) for p, q in zip(used.parameters(), fresh.parameters())), make_opt


def test_gpu_arm_fails_loudly_without_a_device():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"], capture_output=True,
                         text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0 and "no CUDA device" in (out.stderr + out.stdout)
