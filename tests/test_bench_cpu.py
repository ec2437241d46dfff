"""CPU: the reference arm of bench.py (the reference's algorithm on the host cores) prints ONE JSON line with the
contract's keys, and the B200 arm refuses to run without a GPU instead of falling back to anything."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_contract():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1',
                          '--warmup', '0', '--cpu-iters', '4'], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better',
                'scaling', 'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert key in d, key
    assert d['impl'] == 'reference' and d['higher_is_better'] is True and d['value'] > 0
    assert d['config']['workload'].startswith('BASELINE config 2')
    sys.path.insert(0, ROOT)
    import bench
    assert d['config'] == bench.workload_config(1)            # key for key what the B200 arm reports
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1
    assert 'physical_cores' in d['cpu_baseline'] and 'iterations' in d['cpu_baseline']['sample']
    assert d['steps_completed'] == 1 and d['cut_short'] is False
    assert d['cpu_baseline']['value'] == d['value'] == d['e2e']['value']
    assert d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['d2h_bytes_per_step'] == 0


def test_b200_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip('a GPU is present')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '1', '--warmup', '0',
                          '--no-cpu-baseline'], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0
    assert 'no CPU fallback' in (out.stderr + out.stdout)


def test_reference_arm_is_bounded_and_survives_sigterm():
    """The driver gives the reference arm a time slot per N: it must size its sample from a calibration step (not from
    --steps) and still print its JSON line when it is cut short."""
    import signal
    import time
    p = subprocess.Popen([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '400',
                          '--warmup', '1', '--cpu-iters', '60'], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                         text=True, cwd=ROOT)
    time.sleep(12)
    p.send_signal(signal.SIGTERM)
    out, err = p.communicate(timeout=60)
    lines = [ln for ln in out.splitlines() if ln.startswith('{')]
    assert len(lines) == 1, (out[-500:], err[-1500:])
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['cut_short'] is True and d['steps_completed'] < 400


def test_dump_outputs_writes_what_the_timed_call_returned(tmp_path):
    """--dump-outputs: float32 .npy files of an engine.hmc_run result, the sample block reduced to every chain's slots
    0, 32, 64, ... and the last slot (here a CPU stand-in of config 2's shapes with 3 chains)."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from hamiltorch_b200.engine import HMCResult
    C, S, D, ld = 3, bench.S, 6, 8
    g = torch.Generator().manual_seed(0)
    res = HMCResult(torch.randn(C, S, ld, generator=g), (torch.rand(C, S, generator=g) < 0.9).to(torch.uint8),
                    torch.zeros(C, S, dtype=torch.uint8), None, torch.full((C,), 0.05),
                    torch.tensor([3, 0, 7], dtype=torch.int32), D, S)
    res.final_state = torch.randn(C, ld, generator=g)[:, :D]
    bench.dump_outputs(str(tmp_path), res)
    got = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert set(got) == {'samples', 'final_state', 'accepted', 'diverged', 'step_size', 'num_rejected'}
    assert all(a.dtype == np.float32 for a in got.values())
    slots = list(range(0, S, 32)) + [S - 1]
    assert np.array_equal(got['samples'], res.samples[:, slots].numpy())
    assert np.array_equal(got['final_state'], res.final_state.numpy())
    assert np.array_equal(got['accepted'], res.accepted.float().numpy())
    assert got['num_rejected'].tolist() == [3, 0, 7]
    # at config 2's size (256 chains, D = 1024) all files together stay within 64 MiB
    assert 4 * bench.C_PER_GPU * (len(slots) * bench.D + bench.D + 2 * S + 2) <= 64 << 20


def test_host_topology_helpers():
    sys.path.insert(0, ROOT)
    import bench
    h = bench.host_cpus()
    assert h['workers'] >= 1 and h['logical'] >= h['workers']
    assert bench._parse_cpulist('0-3,8,10-11\n') == {0, 1, 2, 3, 8, 10, 11}
    info = bench.bind_to_gpu_numa_node(0)                     # no GPU / NVML here: must not raise
    assert isinstance(info, dict) and 'bound' in info
