"""bench.py: the reference arm's JSON line (CPU) and the CUDA arm's --dump-outputs files (GPU)."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, str(ROOT / 'bench.py'), '--impl', 'reference', '--beam', '2000', '--steps', '1', '--warmup', '0'],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
              'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert k in d, k
    assert d['impl'] == 'reference' and d['higher_is_better'] is True and d['vs_baseline'] is None and d['value'] > 0
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] == 1 and d['cpu_baseline']['value'] == d['value']
    assert d['e2e'] == {'value': d['value'], 'unit': d['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert 'workload' in d['config']


def _reference_arm(steps):
    r = subprocess.run([sys.executable, str(ROOT / 'bench.py'), '--impl', 'reference', '--beam', '2000', '--steps', str(steps), '--warmup', '0'],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout)
    return d, d['value'] * d['ms_per_step'] * 1e-3 * d['steps']  # rate x time = states expanded in the timed steps


def test_steps_sets_the_number_of_timed_steps():
    """Every step is the same deterministic solve, so 4 steps expand exactly 4 times what 1 step does."""
    _, one = _reference_arm(1)
    d, four = _reference_arm(4)
    assert d['steps'] == 4
    assert four == pytest.approx(4 * one, rel=1e-9)


# ------------------------------------------------------------------ --dump-outputs (GPU)
FIELDS = ('level', 'ended', 'frontier', 'expanded', 'generated', 'unique', 'kept', 'goal_rank', 'visited')


def _dumps(tmp_path, *args):
    """bench.py run twice with --dump-outputs -> (first run's arrays, its JSON line); both runs must write the same"""
    lines = []
    for d in ('a', 'b'):
        r = subprocess.run([sys.executable, str(ROOT / 'bench.py'), *args, '--warmup', '0', '--no-parity', '--no-cpu-baseline',
                            '--dump-outputs', str(tmp_path / d)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        lines.append(json.loads(r.stdout.strip().splitlines()[-1]))
    got = {p.stem: np.load(p) for p in (tmp_path / 'a').glob('*.npy')}
    assert sorted(got) == sorted(p.stem for p in (tmp_path / 'b').glob('*.npy'))
    for name, arr in got.items():
        assert arr.dtype == np.float64, name
        assert np.array_equal(arr, np.load(tmp_path / 'b' / f'{name}.npy')), name
    assert sum(p.stat().st_size for p in (tmp_path / 'a').iterdir()) <= 64 << 20
    assert got['levels'].shape[1] == len(FIELDS)
    return got, lines[0]


def _words(rows):
    """records (uint64 columns, or structured 96-byte records) -> the dump's 32-bit words"""
    rows = np.ascontiguousarray(rows)
    return rows.view(np.uint8).reshape(len(rows), -1).view('<u4').astype(np.float64)


def _speedrun_queue(st, lk):
    return _words(np.stack([st['lo'], st['hi'], st['aux'], lk], axis=1).astype(np.uint64))


def _levels_equal(got, infos, fields):
    assert got['levels'].shape[0] == len(infos)
    for f in fields:
        assert got['levels'][:, FIELDS.index(f)].tolist() == [i[f] for i in infos], f


@pytest.mark.gpu
def test_dump_outputs_speedrun(tmp_path):
    """Counters of every level, the full final queue and the API's winning line equal the CPU oracle's search."""
    import oracle
    got, line = _dumps(tmp_path, '--config', 'C1', '--beam', '3000', '--steps', '2')
    assert sorted(got) == ['levels', 'path', 'queue', 'queue_rows']
    assert line['steps'] == 2 and len(line['e2e']['seconds_each_solve_rank0']) == 2
    orc = oracle.Solver(10, use_heuristic=True, heuristic_name='simple', beam_width=3000, policy='stable', noise='const')
    infos = orc.run()
    _levels_equal(got, infos, ('level', 'frontier', 'expanded', 'generated', 'unique', 'kept', 'goal_rank', 'visited'))
    st, lk = orc.level(infos[-1]['level'])
    assert got['queue_rows'].tolist() == list(range(len(st)))
    assert np.array_equal(got['queue'], _speedrun_queue(st, lk))
    p = orc.path()
    assert np.array_equal(got['path'], _words(np.stack([p['lo'], p['hi'], p['aux']], axis=1)))
    orc.close()


@pytest.mark.gpu
def test_dump_outputs_sample_a_large_queue(tmp_path):
    """A final queue over the size budget is dumped as a sorted sample of its ranks, each row the oracle's record."""
    import oracle
    got, _ = _dumps(tmp_path, '--config', 'C3', '--beam', '1000000', '--steps', '1')
    n = int(got['levels'][-1, FIELDS.index('frontier')])
    rows = got['queue_rows'].astype(np.int64)
    assert 0 < len(rows) < n and (np.diff(rows) > 0).all() and rows[0] >= 0 and rows[-1] < n
    assert got['queue'].shape == (len(rows), 8)
    orc = oracle.Solver(15, use_heuristic=True, heuristic_name='aggressive', beam_width=1_000_000, policy='stable', noise='const')
    infos = orc.run()
    _levels_equal(got, infos, ('level', 'frontier', 'expanded', 'generated', 'unique', 'goal_rank', 'visited'))
    st, lk = orc.level(infos[-1]['level'])
    assert np.array_equal(got['queue'], _speedrun_queue(st[rows], lk[rows]))
    orc.close()


@pytest.mark.gpu
def test_dump_outputs_bfs(tmp_path):
    """Exhaustive BFS (no goal, no path): counters of every level and the queue it stops at equal the oracle's."""
    import oracle
    got, _ = _dumps(tmp_path, '--config', 'C2', '--bfs-depth', '4', '--steps', '1')
    assert sorted(got) == ['levels', 'queue', 'queue_rows']
    orc = oracle.Solver(255, use_heuristic=False, heuristic_name='simple', beam_width=0, policy='stable', noise='const')
    infos = [orc.step() for _ in range(4)]
    _levels_equal(got, infos, ('level', 'frontier', 'expanded', 'generated', 'unique', 'kept', 'goal_rank', 'visited'))
    st, lk = orc.level(4)
    assert np.array_equal(got['queue'], _speedrun_queue(st, lk))
    orc.close()


@pytest.mark.gpu
def test_dump_outputs_realistic(tmp_path):
    """Realistic mode (96-byte records): counters of every ply, the final queue and the winning line equal the oracle's."""
    import oracle
    import splendor_rl_gym_b200 as S
    got, _ = _dumps(tmp_path, '--config', 'C5', '--players', '2', '--beam', '2000', '--steps', '1')
    assert sorted(got) == ['levels', 'path', 'queue', 'queue_rows']
    m = S.CardMarket.from_full_deck(shuffle=True, seed=0)
    market = [list(m.tier1_visible + m.tier1_deck), list(m.tier2_visible + m.tier2_deck), list(m.tier3_visible + m.tier3_deck)]
    orc = oracle.RSolver(oracle.make_rconfig(2, 15, 4, market), 2000)
    infos = orc.run()
    # the ply that finds the finished game is not expanded on the GPU: only its size is compared
    _levels_equal({'levels': got['levels'][:-1]}, infos[:-1], ('level', 'frontier', 'expanded', 'generated', 'unique', 'visited'))
    _levels_equal({'levels': got['levels'][-1:]}, infos[-1:], ('level', 'frontier'))
    q = orc.level(infos[-1]['level'])
    assert got['queue_rows'].tolist() == list(range(len(q)))
    assert np.array_equal(got['queue'], _words(q))
    p = orc.path().copy()
    p['link'] = np.uint64((1 << 64) - 1)  # MultiPlayerState.record() carries no parent link
    assert np.array_equal(got['path'], _words(p))
    orc.close()


def test_reference_arm_other_ranks_stay_silent(monkeypatch):
    env = dict(__import__('os').environ, RANK='1', WORLD_SIZE='2')
    r = subprocess.run([sys.executable, str(ROOT / 'bench.py'), '--impl', 'reference', '--beam', '2000', '--steps', '1', '--warmup', '0'],
                       capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ''
