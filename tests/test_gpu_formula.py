"""GPU tests (-m gpu) of formula heuristics (splendor-rl-gym_b200/formula.py, spl_add_formula): scores bit for bit
against the CPU oracle of formulas (tests/formula_oracle.py) in every noise mode; the built-in twins reproduce the
reference's golden runs; new formulas level by level against that oracle on the card-set-grouped level (including its
radix-select fallback), the key-table level and the 'det' tie policy; the drop-in claim of formula.reference();
batches; two gloo ranks on one GPU; engine errors."""
import ctypes as C
import json
import os
import random
import tempfile
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import formula_oracle
import oracle
import splendor_rl_gym_b200 as S
from common import assert_digest, level_digest
from splendor_rl_gym_b200 import HEURISTICS, Formula
from splendor_rl_gym_b200._lib import SplendorB200Error, lib
from splendor_rl_gym_b200.formula import BUILTIN_TWINS
from splendor_rl_gym_b200.sharded import Comm, CudaBackend, DictionaryOverflow, GroupedShardedSolver, ShardedSolver

pytestmark = pytest.mark.gpu

SPL_E_INVALID = -1
FIELDS = ('frontier', 'generated', 'unique', 'kept', 'goal_rank', 'visited')
GOLDEN = Path(__file__).parent / 'golden'

#: negative coefficients, three-factor terms, per-colour features
MIXED = Formula([(-3.5, ('pts', 2.0)), (0.25, ('saved', 0.5), ('cards', 1.1), ('colors', 0.3)), (-7, ('gem_red', 1.5)),
                 (40.0, ('pts', 2.6))])
COLOURS = Formula([(1e-3, ('bonus_white', 2.0), ('bonus_black', 1.0)), (-2.0, ('gems', 0.9)), (4.0, ('resources', 0.45)),
                   (1.5, ('gem_white', 0.0), ('bonus_green', 3.0), ('gem_blue', 0.7)), (90.0, ('pts', 2.2))])
#: so many distinct scores per level that the score dictionary of the cut (2048 entries) overflows
MANY = Formula([(1.0, ('saved', 0.5)), (30.0, ('pts', 2.1)), (1e-3, ('gems', 1.3), ('cards', 0.9)),
                (1e-6, ('bonus_red', 1.1), ('gem_blue', 0.8), ('bonus_white', 1.7))])
NEW = {'mixed': MIXED, 'colours': COLOURS, 'many': MANY}


@pytest.fixture(scope='module')
def eng():
    return S.Engine.get(0)


@pytest.fixture(scope='module')
def states():
    s = oracle.Solver(99, use_heuristic=False)
    s.run(max_levels=6)
    bfs6 = s.level(6)[0]
    assert len(bfs6) == 166_688
    rng = random.Random(11)
    edge = np.zeros(2000, oracle.STATE_DTYPE)
    for i in range(len(edge)):
        top = i % 2 == 0
        gems = [rng.randint(0, 2) for _ in range(5)]
        edge[i] = oracle.pack_state(tuple(sorted(rng.sample(range(90), rng.choice([0, 3, 45, 90])))),
                                    tuple(31 if top else rng.randint(0, 31) for _ in range(5)), tuple(gems),
                                    255 if top else rng.randint(0, 255), 65535 if top else rng.randint(0, 65535))[0]
    return np.concatenate([bfs6, edge])


def _bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


# ------------------------------------------------------------------ spl_score / spl_score_rows
@pytest.mark.parametrize('noise', ['const', 'hash', 'mt'])
def test_scores_bit_exact_vs_oracle(eng, states, noise):
    keys = np.stack([states['lo'], states['hi']], axis=1)
    k, a = eng.to_device(keys, states['aux'])
    rows = torch.stack([k[:, 0], k[:, 1], a, torch.zeros_like(a)], 1).contiguous()
    draws = np.random.default_rng(5).integers(1, 101, len(states)).astype(np.uint8)
    for f in [*NEW.values(), *BUILTIN_TWINS.values()]:
        if noise == 'mt':
            got = CudaBackend(eng).score(f, 'mt', rows, torch.from_numpy(draws).to(eng.tdev)).cpu().numpy()
            want = formula_oracle.score(states, f, draws=draws)
        else:
            got = eng.score(f, k, a, noise).cpu().numpy()
            want = formula_oracle.score(states, f, noise)
            assert (_bits(CudaBackend(eng).score(f, noise, rows).cpu().numpy()) == _bits(want)).all(), f
        assert (_bits(got) == _bits(want)).all(), f
    assert (formula_oracle.score(states, MIXED) < 0).any()  # negative totals
    st = S.State.from_record(int(states[-2]['lo']), int(states[-2]['hi']), int(states[-2]['aux']))
    assert _bits([MIXED(st)])[0] == _bits(formula_oracle.score(states[-2:-1], MIXED))[0]


# ------------------------------------------------------------------ the twins reproduce the reference
@pytest.fixture
def twins(monkeypatch):
    for name, f in BUILTIN_TWINS.items():
        monkeypatch.setitem(HEURISTICS, f'twin_{name}', f)
    return {name: f'twin_{name}' for name in BUILTIN_TWINS}


def test_twins_reproduce_golden_beam_runs(eng, golden, twins):
    assert len(golden['beam_runs']) == 37
    for run in golden['beam_runs']:
        what = f"twin {run['base']}@{run['policy']}/{run['noise']} goal={run['goal']} beam={run['beam']}"
        k, a = S.State.newgame().record()
        sol = eng.solver(k, a, run['goal'], True, BUILTIN_TWINS[run['base']], run['beam'], run['policy'], run['noise'])
        for want in run['levels']:
            gi = sol.step()
            assert (gi['frontier'], gi['generated'], gi['unique']) == (want['frontier'], want['generated'], want['unique']['n']), what
            if not gi['ended']:
                fr = sol.frontier().cpu().numpy().view(np.uint64)
                assert_digest(level_digest(fr[:, 0], fr[:, 1], fr[:, 2], fr[:, 3]), want['kept'], f"{what} level {want['level']}")
        assert gi['ended'] and gi['visited'] == run['visited'], what
        sol.close()
        path = S.State.newgame().solve(goal_pts=run['goal'], use_heuristic=True, heuristic_name=twins[run['base']],
                                       beam_width=run['beam'], verbose=False, tie_policy=run['policy'], noise=run['noise'])
        assert [repr(s) for s in path] == [p['repr'] for p in run['path']], what
        assert [(s.saved, s.pts, list(s.bonus)) for s in path] == [(p['saved'], p['pts'], p['bonus']) for p in run['path']], what


def test_twins_reproduce_seeded_reference(golden, twins):
    runs = [r for r in golden['mt_runs'] if r['mode'] == 'speedrun']
    assert runs
    for run in runs:
        what = f"twin mt {run['heuristic']} seed={run['seed']}"
        random.seed(run['seed'])
        stats = []
        line = S.State.newgame().solve(goal_pts=run['goal'], use_heuristic=True, heuristic_name=twins[run['heuristic']],
                                       beam_width=run['beam'], verbose=False, noise='mt', stats=stats)
        assert [repr(s) for s in line] == [p['repr'] for p in run['path']], what
        assert [random.randint(1, 100) for _ in range(4)] == run['after'], what
        for info, want in zip(stats, run['levels']):
            assert info['frontier'] == want['frontier'], what


# ------------------------------------------------------------------ new formulas vs the oracle, level by level
def _vs_oracle(eng, f, beam, policy='stable', noise='const', goal=15, identity='key'):
    k, a = S.State.newgame().record()
    sol = eng.solver(k, a, goal, True, f, beam, policy, noise, identity=identity)
    orc = formula_oracle.Solver(goal, f, beam_width=beam, policy=policy, noise=noise, identity=identity)
    what = f'{f} beam={beam} {policy}/{noise}/{identity}'
    try:
        while True:
            gi, oi = sol.step(), orc.step()
            for fld in FIELDS:
                assert gi[fld] == oi[fld], (what, fld, gi, oi)
            if gi['ended']:
                assert orc.done, what
                break
            fr = sol.frontier().cpu().numpy().view(np.uint64)
            st, lk = orc.level(oi['level'] + 1)
            assert fr.tobytes() == np.stack([st['lo'], st['hi'], st['aux'], lk], 1).tobytes(), (what, gi['level'])
        ranks, ords = sol.path()
        want = orc.path()
        line = [np.zeros(1, oracle.STATE_DTYPE)]
        line[0][0] = want[0]
        for o in ords:
            line.append(oracle.expand(line[-1])[o:o + 1])
        assert np.concatenate(line).tobytes() == want.tobytes(), what
        return sol.infos
    finally:
        sol.close()
        orc.close()


@pytest.mark.parametrize('name,beam,noise', [('mixed', 1000, 'const'), ('colours', 1000, 'hash'), ('many', 1000, 'hash'),
                                             ('mixed', 300_000, 'const'), ('many', 300_000, 'const')])
def test_grouped_level_vs_oracle(eng, name, beam, noise):
    infos = _vs_oracle(eng, NEW[name], beam, noise=noise)
    if name == 'many' and beam == 300_000:
        assert max(i['unique'] for i in infos) > 300_000  # levels that need the cut (the dictionary overflows there)


@pytest.mark.parametrize('name', ['mixed', 'many'])
def test_key_table_level_vs_oracle(eng, name, monkeypatch):
    monkeypatch.setenv('SPL_NO_GROUPED', '1')
    _vs_oracle(eng, NEW[name], 20_000, noise='hash')
    _vs_oracle(eng, NEW[name], 5_000, identity='pyhash')
    eng.set_identity('key')


@pytest.mark.parametrize('name,beam', [('mixed', 2_000), ('many', 50_000), ('colours', 10_000)])
def test_det_ties_vs_oracle(eng, name, beam):
    _vs_oracle(eng, NEW[name], beam, policy='det', noise='const')


def _python_beam_line(f, goal, beam):
    """the reference's solve() loop (src/solver.py:426-464) over oracle.expand, scored by f.reference() with the global
    `random` -- the drop-in claim without the reference itself"""
    h = f.reference()
    key = lambda r: (int(r['lo']), int(r['hi']))  # noqa: E731
    root = oracle.pack_state((), (0,) * 5, (0,) * 5, 0, 0)[0]
    trail = {key(root): None}
    queue = [root]
    while queue:
        nxt = []
        for st in queue:
            if (int(st['aux']) >> 16) & 0xff >= goal:
                line = [st]
                while trail[key(line[-1])] is not None:
                    line.append(trail[key(line[-1])])
                return [oracle.unpack_state(r) for r in reversed(line)]
            for ch in oracle.expand(st):
                if key(ch) not in trail:
                    trail[key(ch)] = st
                    nxt.append(ch)

        def score(r):
            u = oracle.unpack_state(r)
            return h(SimpleNamespace(cards=u['cards'], gems=u['gems'], bonus=u['bonus'], pts=u['pts'], saved=u['saved']))
        queue = sorted(nxt, key=score, reverse=True)[:beam]
    return None


@pytest.mark.parametrize('name', ['mixed', 'many'])
def test_reference_function_drop_in_mt(eng, name, monkeypatch):
    f, goal, beam = NEW[name], 8, 400
    random.seed(1234)
    want = _python_beam_line(f, goal, beam)
    after = [random.randint(1, 100) for _ in range(3)]
    random.seed(1234)
    line = S.State.newgame().solve(goal_pts=goal, use_heuristic=True, heuristic_name=f, beam_width=beam, verbose=False,
                                   noise='mt')
    assert [(s.cards, s.gems, s.pts, s.saved) for s in line] == [(w['cards'], w['gems'], w['pts'], w['saved']) for w in want]
    assert [random.randint(1, 100) for _ in range(3)] == after
    # the key-table level with the reference's hash identity and the reference's noise stream
    monkeypatch.setenv('SPL_NO_GROUPED', '1')
    random.seed(1234)
    line = S.State.newgame().solve(goal_pts=goal, use_heuristic=True, heuristic_name=f, beam_width=beam, verbose=False,
                                   noise='mt', identity='pyhash')
    assert [(s.cards, s.gems, s.pts, s.saved) for s in line] == [(w['cards'], w['gems'], w['pts'], w['saved']) for w in want]
    eng.set_identity('key')


# ------------------------------------------------------------------ batches
def test_solve_many_mixed_batch(eng, monkeypatch):
    monkeypatch.setitem(HEURISTICS, 'mixed', MIXED)
    roots = [S.State.newgame()] * 6
    names = ['mixed', 'aggressive', COLOURS, MANY, 'simple', 'mixed']
    kinds = [True, True, True, True, False, True]
    beams = [2_000, 3_000, 1_000, 5_000, 1, 500]
    goals = [12, 12, 10, 12, 4, 9]
    lines = S.State.solve_many(roots, goals, use_heuristic=kinds, heuristic_name=names, beam_width=beams, noise='hash')
    for g in range(len(roots)):
        one = roots[g].solve(goals[g], use_heuristic=kinds[g], heuristic_name=names[g], beam_width=beams[g], verbose=False,
                             noise='hash')
        assert [(s.cards, s.gems, s.pts, s.saved) for s in lines[g]] == [(s.cards, s.gems, s.pts, s.saved) for s in one], g


def test_solve_many_sweep_of_1024_formulas(eng):
    sweep = [Formula([(100.0 + i, ('pts', 2.0 + (i % 16) / 20)), (1.0 + i / 64, ('saved', 0.5)), (-0.5, ('gem_green', 1.0))])
             for i in range(1024)]
    lines = S.State.solve_many([S.State.newgame()] * 1024, 8, use_heuristic=True, heuristic_name=sweep, beam_width=200)
    for i in (0, 17, 511, 1023):
        one = S.State.newgame().solve(8, use_heuristic=True, heuristic_name=sweep[i], beam_width=200, verbose=False)
        assert [(s.cards, s.gems, s.pts, s.saved) for s in lines[i]] == [(s.cards, s.gems, s.pts, s.saved) for s in one], i
    assert all(line[-1].pts >= 8 for line in lines)


# ------------------------------------------------------------------ engine errors
def test_engine_errors_and_limits():
    eng = S.Engine(0)
    other = S.Engine(0)
    try:
        fid = eng.heuristic_id(MIXED)
        assert fid == 256 and eng.heuristic_id(MIXED) == fid  # registered once
        k, a = eng.to_device(np.zeros((1, 2), np.uint64), np.zeros(1, np.uint64))
        out = torch.empty(1, dtype=torch.float64, device=eng.tdev)
        for h in (fid + 1, 256 + 4095):  # unregistered here; foreign (registered on `eng` only)
            assert lib.spl_score(eng._h, h, 0, k.data_ptr(), a.data_ptr(), 1, out.data_ptr(), None) == SPL_E_INVALID
        assert lib.spl_score(other._h, fid, 0, k.data_ptr(), a.data_ptr(), 1, out.data_ptr(), None) == SPL_E_INVALID
        h = C.c_void_p()
        key = S._lib.Key(0, 0)
        assert lib.spl_solver_create(other._h, C.byref(key), 0, 15, 1, fid, 100, 0, 0, 1, C.byref(h)) == SPL_E_INVALID
        assert lib.spl_gs_create(other._h, 0, 1, C.byref(key), 0, 15, fid, 100, 0, 1, C.byref(h)) == SPL_E_INVALID
        with pytest.raises(SplendorB200Error, match='SPL_E_INVALID'):
            other.sbatch_solver(np.zeros((1, 4), np.uint64), [15], [True], [fid], [100])
        # ids outside the formula range keep their meaning: the fallback to simple
        assert other.score(4, k, a).item() == other.score('simple', k, a).item()
        # the formula limit: 4096 per context
        for i in range(1, 4096):
            eng.heuristic_id(Formula([(float(i), ('gem_white', 1.0))]))
        with pytest.raises(SplendorB200Error, match='SPL_E_CAPACITY'):
            eng.heuristic_id(Formula([(-1.0, ('gem_white', 1.0))]))
        # the table limit: 256 MiB of power tables (512 KiB per saved exponent)
        line2 = S.State.newgame().solve(10, use_heuristic=True, heuristic_name=MIXED, beam_width=500, verbose=False, engine=other)
        with pytest.raises(SplendorB200Error, match='SPL_E_CAPACITY'):
            for i in range(600):
                other.heuristic_id(Formula([(1.0, ('saved', 0.001 * (i + 1)))]))
        # both engines still work, with the formulas they hold
        line = S.State.newgame().solve(10, use_heuristic=True, heuristic_name=MIXED, beam_width=500, verbose=False, engine=eng)
        line3 = S.State.newgame().solve(10, use_heuristic=True, heuristic_name=MIXED, beam_width=500, verbose=False, engine=other)
        assert [repr(s) for s in line] == [repr(s) for s in line2] == [repr(s) for s in line3] and line[-1].pts >= 10
    finally:
        eng.close()
        other.close()


# ------------------------------------------------------------------ two gloo ranks on one GPU
def _entry(rank, world, init_file, out_file, fn, args):
    dist.init_process_group('gloo', init_method=f'file://{init_file}', rank=rank, world_size=world)
    try:
        eng = S.Engine(0)
        comm = Comm(eng.tdev)
        out = fn(eng, comm, *args)
        peer = getattr(eng, '_peer_recv', None)
        if peer is not None:
            peer.release()
        eng.close()
        if rank == 0:
            Path(out_file).write_text(json.dumps(out))
    finally:
        dist.destroy_process_group()


def _spawn(world, fn, *args):
    with tempfile.TemporaryDirectory() as d:
        init_file, out_file = os.path.join(d, 'init'), os.path.join(d, 'out')
        mp.spawn(_entry, args=(world, init_file, out_file, fn, args), nprocs=world, join=True)
        return json.loads(Path(out_file).read_text())


def _solve_ranks(eng, comm):
    calls = dict(grouped=0, key=0, overflow=0)
    g_step, k_step = GroupedShardedSolver.step, ShardedSolver.step

    def grouped_step(self):
        calls['grouped'] += 1
        try:
            return g_step(self)
        except DictionaryOverflow:
            calls['overflow'] += 1
            raise

    def key_step(self):
        calls['key'] += 1
        return k_step(self)

    GroupedShardedSolver.step, ShardedSolver.step = grouped_step, key_step
    HEURISTICS['mixed'], HEURISTICS['many'] = MIXED, MANY
    out = {}
    try:
        for name, beam in (('mixed', 20_000), ('many', 40_000)):
            for c in calls:
                calls[c] = 0
            line = S.State.newgame().solve(15, use_heuristic=True, heuristic_name=name, beam_width=beam, verbose=False,
                                           engine=eng)
            if comm.rank == 0:
                orc = formula_oracle.Solver(15, NEW[name], beam_width=beam)
                orc.run()
                want = [tuple(oracle.unpack_state(w)[f] for f in ('cards', 'bonus', 'gems', 'pts', 'saved')) for w in orc.path()]
                assert [(s.cards, s.bonus, s.gems, s.pts, s.saved) for s in line] == want, name
                orc.close()
            out[name] = dict(calls)
    finally:
        GroupedShardedSolver.step, ShardedSolver.step = g_step, k_step
        del HEURISTICS['mixed'], HEURISTICS['many']
    return out


def test_state_solve_two_ranks_vs_oracle():
    out = _spawn(2, _solve_ranks)
    assert out['mixed']['grouped'] > 0 and out['mixed']['key'] == 0 and out['mixed']['overflow'] == 0
    assert out['many']['overflow'] == 1 and out['many']['key'] > 0  # the many-score formula falls back to the key-sharded driver
