"""bench.py contract on the CPU: the reference arm (the oracle port timed on the host cores, a bounded sample per step) prints
ONE JSON line with the keys the driver reads, on the same metric / unit / workload name as the GPU arm."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0'],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline',
              'dtype', 'data', 'config', 'impl', 'cpu_baseline', 'e2e'):
        assert k in d, k
    assert d['impl'] == 'reference' and d['metric'] == 'genomes/hour' and d['unit'] == 'genomes/hour'
    assert d['higher_is_better'] is True and d['vs_baseline'] is None and d['value'] > 0
    assert d['cpu_baseline']['kind'] in ('port', 'hmmer') and d['cpu_baseline']['cores'] >= 1 and d['cpu_baseline']['value'] == d['value']
    assert d['e2e'] == {"value": d['value'], "unit": d['unit'], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    sys.path.insert(0, ROOT)
    import bench
    assert d['config']['workload'] == bench.workload_name(3, bench.total_model_positions(bench.model_db()))
    assert 'no extrapolation' in d['cpu_baseline']['sample'] and d['cpu_baseline']['gcups_per_core'] > 0


def test_dump_outputs_fields_and_sample(tmp_path):
    """--dump-outputs: one float32 / float64 file per field, a fixed seeded sample of a table too large for the budget."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from checkm_b200.engine import HIT_DTYPE
    from checkm_b200.resultsParser import QA_DTYPE
    hits = np.zeros(400000, dtype=HIT_DTYPE)
    hits['seq'] = np.arange(len(hits))
    hits['dom_score'] = np.linspace(-5.0, 50.0, len(hits), dtype=np.float32)
    qa = np.zeros(32, dtype=QA_DTYPE)
    qa['counts'][:, 1] = 7
    qa['completeness'] = np.arange(32) / 3.0
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), {'hits': hits, 'qa': qa})
    files = sorted(os.listdir(tmp_path / 'a'))
    assert files == sorted(os.listdir(tmp_path / 'b'))
    assert set(files) == {'hits_%s.npy' % f for f in HIT_DTYPE.names + ('row',)} | {'qa_%s.npy' % f for f in QA_DTYPE.names + ('row',)}
    assert sum(os.path.getsize(tmp_path / 'a' / f) for f in files) <= 64 * 1000 * 1000
    for f in files:
        a, b = np.load(tmp_path / 'a' / f), np.load(tmp_path / 'b' / f)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), f
    rows = np.load(tmp_path / 'a' / 'hits_row.npy')
    assert 0 < len(rows) < len(hits) and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(tmp_path / 'a' / 'hits_seq.npy'), rows)
    score = np.load(tmp_path / 'a' / 'hits_dom_score.npy')
    assert score.dtype == np.float32 and np.array_equal(score, hits['dom_score'][rows.astype(np.int64)])
    assert np.array_equal(np.load(tmp_path / 'a' / 'qa_row.npy'), np.arange(32))
    assert np.array_equal(np.load(tmp_path / 'a' / 'qa_counts.npy'), qa['counts'])
    assert np.array_equal(np.load(tmp_path / 'a' / 'qa_completeness.npy'), qa['completeness'])


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK='1', LOCAL_RANK='1', WORLD_SIZE='2')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2', '--steps', '1', '--warmup', '0'],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ''
