"""bench.py end to end on the CPU (tests/bench_dry_run.py: inert CUDA stand-ins, emulated kernels, a tiny clip): both
timed arms, the look-ahead extension arm, the in-run parity check against the oracle, the CPU baseline and the JSON
assembly all execute, exactly one JSON line reaches stdout and it carries every key the contract names."""
import json
import os
import subprocess
import sys

from tests.conftest import ROOT

REQUIRED = ['metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
            'vs_baseline', 'dtype', 'data', 'config', 'clocks', 'e2e', 'gpu_launches', 'roofline', 'cpu_baseline',
            'parity_check', 'latency_ms']


def _run(*extra):
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'bench_dry_run.py'), '--steps', '6', '--warmup', '3',
                        *extra], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    return json.loads(lines[0]), r.stderr


def test_bench_control_flow_runs_and_prints_one_json_line():
    line, err = _run()
    for k in REQUIRED:
        assert k in line, k
    assert line['steps'] == 6 and line['warmup'] == 3 and line['n_gpus'] == 1 and line['higher_is_better'] is True
    assert line['untimed_steps_before_timed_region'] >= 11      # graphs requested: every capture variant exists
    assert line['e2e']['h2d_bytes_per_step'] > 0 and line['e2e']['d2h_bytes_per_step'] > 0
    assert line['config']['workload'].startswith('tiny')
    assert set(line['config']) == {'workload', 'resolution', 'objects', 'tokens_per_frame', 'memory_tokens', 'top_k',
                                   'mem_every', 'streams', 'parallelism', 'l2', 'weights', 'precision'}
    assert line['cpu_baseline']['kind'] == 'port' and line['cpu_baseline']['value'] > 0
    assert line['latency_ms']['frames'] == 6 and line['latency_ms']['p99'] >= line['latency_ms']['p50'] > 0
    pc = line['parity_check']
    assert 'error' not in pc, pc
    assert pc['within_1e-3'] and pc['max_abs_logit_diff'] < 1e-3 and pc['queries'] > 0
    assert line['build']['cudnn_allow_tf32'] is False and line['build']['glue_dispatch']['table']
    la = line['with_encoder_lookahead']
    assert la and la['value'] > 0 and la['e2e'] > 0
    assert line['roofline'] is not None and line['roofline']['achieved'] > 0


def test_bench_drop_in_only_and_no_checks():
    line, err = _run('--no-lookahead', '--no-cpu-baseline', '--no-parity-check')
    assert line['with_encoder_lookahead'] is None and line['cpu_baseline'] is None and line['parity_check'] is None
    assert line['value'] > 0 and line['e2e']['value'] > 0


def test_bench_dumps_the_last_timed_step_and_repeats_it(tmp_path):
    """--dump-outputs: the probabilities InferenceCore.step returned in the last timed step, float32, the same from run to
    run with the same arguments (seeded inputs); --steps sets the number of timed steps."""
    import numpy as np
    outs = []
    for run, steps in (('a', 5), ('b', 5), ('c', 4)):
        d = tmp_path / run
        line, err = _run('--no-lookahead', '--no-cpu-baseline', '--no-parity-check', '--steps', str(steps),
                         '--dump-outputs', str(d))
        assert line['steps'] == steps and line['latency_ms']['frames'] == steps
        assert sorted(os.listdir(d)) == ['prob.npy']
        outs.append(np.load(d / 'prob.npy'))
    a, b, c = outs
    assert a.dtype == np.float32 and a.ndim == 3 and a.shape[0] == 1 + line['config']['objects']
    assert np.isfinite(a).all() and np.allclose(a.sum(0), 1, atol=1e-4)
    assert np.array_equal(a, b)
    assert not np.array_equal(a, c)             # one timed step fewer: another frame's output
