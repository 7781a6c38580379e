"""bench.py --dump-outputs: what the timed path returned in its last timed step, within 64 MB, the same for the same arguments."""
import importlib.util
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SR = 48000.0


def _bench():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def _run(tmp_path, *args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(tmp_path / "out")],
                          capture_output=True, text=True, cwd=ROOT, timeout=900)


@pytest.mark.parametrize("shape", [(2, 48000), (16384 * 2, 48000), (1, 10 << 20), (3, 4 << 20)])
def test_dump_sample_fits_the_budget_and_is_fixed(shape):
    bench = _bench()
    budget = bench.DUMP_BYTES // 2
    r, c = bench.dump_sample(shape, budget)
    r2, c2 = bench.dump_sample(shape, budget)
    assert np.array_equal(r, r2) and np.array_equal(c, c2)
    assert len(r) * len(c) * 4 <= budget and len(r) >= 1 and len(c) >= 1
    assert np.all(np.diff(r) > 0) and np.all(np.diff(c) > 0) and r[-1] < shape[0] and c[-1] < shape[1]
    if shape[0] * shape[1] * 4 <= budget:
        assert len(r) == shape[0] and len(c) == shape[1]
    elif shape[1] * 4 <= budget:
        assert len(c) == shape[1]       # whole rows are kept while one fits


def test_steps_must_be_positive(tmp_path):
    r = _run(tmp_path, "--impl", "reference", "--steps", "0")
    assert r.returncode == 2 and "--steps" in r.stderr


def test_reference_arm_dumps_its_last_mix(tmp_path):
    from fundsp_b200 import workloads
    from oracle import oracle_bank_render
    r = _run(tmp_path, "--impl", "reference", "--workload", "noise_svf", "--voices", "8", "--seconds", "0.01", "--steps", "2", "--warmup", "0")
    assert r.returncode == 0, r.stderr[-2000:]
    got = np.load(tmp_path / "out" / "mix.npy")
    _, want = oracle_bank_render(workloads.build("noise_svf", 8), SR, 480, per_voice=False, mix=True)
    assert got.dtype == np.float32 and np.array_equal(got, want)


@pytest.mark.gpu
def test_gpu_arm_dumps_the_last_timed_step(tmp_path):
    """Warm-up max(3, W) device + host-buffer steps, then K timed steps, all on one bank: the dump is samples [(2 max(3, W) + K - 1) n,
    (2 max(3, W) + K) n) of the bank's output from its construction-time state."""
    from fundsp_b200 import workloads
    from oracle import oracle_bank_render
    V, n, K = 256, 4800, 2
    r = _run(tmp_path, "--workload", "noise_svf", "--voices", str(V), "--seconds", str(n / SR), "--steps", str(K), "--warmup", "1", "--per-voice")
    assert r.returncode == 0, r.stderr[-2000:]
    mix, voices = np.load(tmp_path / "out" / "mix.npy"), np.load(tmp_path / "out" / "voices.npy")
    total = (2 * 3 + K) * n
    want_v, want_m = oracle_bank_render(workloads.build("noise_svf", V), SR, total, per_voice=True, mix=True)
    assert voices.shape == (V, n) and np.array_equal(voices, want_v[:, 0, -n:])
    assert mix.shape == (1, n) and np.abs(mix - want_m[:, -n:]).max() <= 1e-5 * np.abs(want_m).max()
