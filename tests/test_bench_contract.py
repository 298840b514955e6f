"""bench.py contract checks that need no GPU: the reference arm runs here (CPU port of the reference path) and prints
exactly one JSON line with the agreed keys; the bench lines committed under profiles/ carry every key the round-end
driver reads (roofline / cpu_baseline / e2e / clocks / gpu_launches)."""
import glob
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline',
             'dtype', 'data', 'config'}


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, THA4_CPU_THREADS='8')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '3'],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and BASE_KEYS <= set(d)
    assert d['metric'] == '512x512 RGBA frames/sec' and d['unit'] == 'frames/s' and d['higher_is_better'] is True
    assert d['value'] > 0 and d['cpu_baseline']['kind'] in ('port', 'reference') and d['cpu_baseline']['cores'] >= 1
    assert d['e2e'] == {'value': d['value'], 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}


def test_dump_outputs_small_in_full_large_as_a_repeatable_sample(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import numpy
    import torch
    import bench
    small = [('a', torch.arange(12.0).reshape(3, 4)), ('b', torch.ones(5, dtype=torch.float64))]
    bench.dump_outputs(str(tmp_path / 'small'), small)
    assert numpy.array_equal(numpy.load(tmp_path / 'small' / 'a.npy'), small[0][1].numpy())
    assert numpy.load(tmp_path / 'small' / 'b.npy').dtype == numpy.float32
    monkeypatch.setattr(bench, 'DUMP_BUDGET_BYTES', 4 * 1000)
    large = [('x', torch.randn(3000)), ('y', torch.randn(2, 500))]
    for d in ('r1', 'r2'):
        bench.dump_outputs(str(tmp_path / d), large)
    sizes = 0
    for name, t in large:
        a, b = (numpy.load(tmp_path / d / (name + '.npy')) for d in ('r1', 'r2'))
        assert numpy.array_equal(a, b) and numpy.isin(a, t.numpy()).all()
        sizes += a.size
    assert 900 <= sizes <= 1000


def test_round2_default_bench_line_has_the_sub_objects():
    """The round-2 default line (BASELINE configs[1]) carries the other configs as sub-objects and the >= 30x denominator."""
    f = os.path.join(ROOT, 'profiles', 'r02_final_bench_default.json')
    d = json.load(open(f))
    assert BASE_KEYS <= set(d) and d['n_gpus'] == 1 and d['gpu_launches'] > 0
    assert d['e2e']['value'] > 0 and d['e2e']['d2h_bytes_per_step'] == 512 * 512 * 4       # the uint8 frame
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['value'] > 0
    for key in ('pose_sweep_512', 'distill', 'student_b64', 'torch_cuda_eager'):
        assert key in d, key
    assert d['pose_sweep_512']['scaling'] == 'strong' and d['pose_sweep_512']['frames_total'] == 512
    assert d['distill']['steps_per_s'] > 0 and d['torch_cuda_eager_fps'] > 0
    assert d['cuda_graphs']['replays'] > 0 and d['cuda_graphs']['failures'] == 0
    for r in (d['roofline'], d['roofline_tail']):
        assert r['bound'] in ('hbm', 'tensor') and abs(r['frac'] - r['achieved'] / r['peak']) < 1e-9
    ref = json.load(open(os.path.join(ROOT, 'profiles', 'r02_final_bench_reference_arm.json')))
    assert ref['impl'] == 'reference' and ref['config'] == d['config'], 'the two arms must print the same config'


def test_round2_final_bench_line_if_committed():
    """The bench line of the end of round 2 (second half), when its evidence run made it into profiles/."""
    f = os.path.join(ROOT, 'profiles', 'r02b_final_bench_default.json')
    if not os.path.exists(f):
        return
    d = json.load(open(f))
    assert BASE_KEYS <= set(d) and d['n_gpus'] == 1 and d['gpu_launches'] > 0 and d['value'] > 0
    assert d['e2e']['value'] > 0 and d['e2e']['d2h_bytes_per_step'] == 512 * 512 * 4
    for key in ('pose_sweep_512', 'distill', 'student_b64', 'torch_cuda_eager', 'roofline', 'roofline_tail', 'cpu_baseline', 'clocks'):
        assert key in d, key
    assert not set(d['clocks']['reasons']) & {'hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown'}


def test_committed_bench_lines_are_complete():
    files = sorted(glob.glob(os.path.join(ROOT, 'profiles', 'r01_final_bench_*.json')))
    assert files, 'round-1 bench lines missing from profiles/'
    seen_default = False
    for f in files:
        d = json.load(open(f))
        if d.get('impl') in ('reference', 'torch_cuda_eager'):
            continue
        assert BASE_KEYS <= set(d), (f, BASE_KEYS - set(d))
        assert d['gpu_launches'] > 0 and d['e2e']['value'] > 0 and d['e2e']['h2d_bytes_per_step'] > 0, f
        assert d['clocks']['sm_mhz'] and not set(d['clocks']['reasons']) & {'hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown'}, f
        r = d['roofline']
        assert r['bound'] in ('hbm', 'tensor') and r['unit'] in ('GB/s', 'TFLOP/s') and r['peak'] > 0, f
        if r['achieved'] is not None:
            assert abs(r['frac'] - r['achieved'] / r['peak']) < 1e-9, f
        if os.path.basename(f) == 'r01_final_bench_teacher_b1.json':
            seen_default = True
            assert d['n_gpus'] == 1 and d['cpu_baseline']['value'] > 0 and d['cpu_baseline']['kind'] == 'port'
            assert d['roofline_tail']['bound'] == 'hbm'
    assert seen_default
