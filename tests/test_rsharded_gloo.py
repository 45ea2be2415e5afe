"""CPU tests of the key-sharded driver in realistic mode (RShardedSolver): world 2 and 3 over gloo, compute primitives
replaced by tests/rfake_backend.py, every level and the winning line compared with the CPU oracle's realistic solver."""
import json
import os
import sys
import tempfile
from pathlib import Path

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = Path(__file__).resolve().parent.parent
for p in (str(ROOT), str(ROOT / 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

RUNS = json.loads((ROOT / 'tests' / 'golden' / 'realistic_runs.json').read_text())


def _ocfg(players, goal, seed, noise='const'):
    run = next(r for r in RUNS if (r['players'], r['seed']) == (players, seed))
    m = run['market']
    return __import__('oracle').make_rconfig(players, goal, run['gems_per_color'], [m['t1'], m['t2'], m['t3']], noise)


def _worker(rank, world, init_file, case, out_file):
    import oracle
    from rfake_backend import RFakeBackend
    from splendor_rl_gym_b200.sharded import Comm, RShardedSolver
    dist.init_process_group('gloo', init_method=f'file://{init_file}', rank=rank, world_size=world)
    try:
        players, goal, seed, beam, block, noise = case
        cfg = _ocfg(players, goal, seed, noise)
        sol = RShardedSolver(RFakeBackend(cfg), Comm(torch.device('cpu')), beam, block_parents=block)
        orc = oracle.RSolver(cfg, beam)
        rounds = []
        keep_all = 0
        while True:
            gi, oi = sol.step(), orc.step()
            fields = ('frontier', 'goal_rank') if gi['ended'] else ('frontier', 'expanded', 'generated', 'unique', 'kept', 'goal_rank', 'visited')
            for f in fields:
                assert gi[f] == oi[f], (rank, f, gi, oi)
            rounds.append(-(-(-(-gi['frontier'] // block)) // world))
            if gi['ended']:
                assert orc.done
                break
            keep_all += gi['unique'] <= beam
            fr = sol.gather_frontier().numpy()
            assert fr.tobytes() == orc.level(oi['level'] + 1).tobytes(), (rank, gi['level'])
        # the winning line: replay the ordinals from the root and compare with the oracle's path, record by record
        ranks, ords = sol.path()
        want = orc.path()
        assert len(ords) == len(want) - 1
        rec = oracle.r_root(cfg)[0]
        got = [oracle.rident_bytes(rec, players)]
        for o in ords:
            rec = oracle.r_expand(cfg, rec)[o]
            got.append(oracle.rident_bytes(rec, players))
        assert got == [oracle.rident_bytes(r, players) for r in want]
        assert ranks[-1] == orc.infos[-1]['goal_rank']
        if rank == 0:
            Path(out_file).write_text(json.dumps(dict(levels=len(sol.infos), max_rounds=max(rounds), keep_all=keep_all)))
    finally:
        dist.destroy_process_group()


def _worker_turn_limit(rank, world, init_file, case, out_file):
    """the turn limit, lowered to `limit` levels: the search stops after cutting level `limit` (as spl_rsolver does at
    level 1000) and the line ends at the last state of that level's queue, walked back through the links"""
    import oracle
    from rfake_backend import RFakeBackend
    from splendor_rl_gym_b200.sharded import Comm, RShardedSolver
    dist.init_process_group('gloo', init_method=f'file://{init_file}', rank=rank, world_size=world)
    try:
        players, goal, seed, beam, block, limit = case

        class Limited(RShardedSolver):
            TURN_LIMIT = limit

        cfg = _ocfg(players, goal, seed)
        sol = Limited(RFakeBackend(cfg), Comm(torch.device('cpu')), beam, block_parents=block)
        orc = oracle.RSolver(cfg, beam)
        for lv in range(limit + 1):
            gi, oi = sol.step(), orc.step()
            for f in ('frontier', 'expanded', 'generated', 'unique', 'kept', 'visited'):
                assert gi[f] == oi[f], (rank, f, gi, oi)
            assert gi['ended'] == (lv == limit) and not orc.done, (rank, gi)
        assert sol.ended and sol.level == limit and sol.goal_rank == gi['frontier'] - 1
        ranks, ords = sol.path()
        assert len(ords) == limit and ranks[-1] == gi['frontier'] - 1
        want, r = [], ranks[-1]
        for lv in range(limit, -1, -1):  # the oracle's queues walked back from the same state
            rec = orc.level(lv)[r]
            want.append(oracle.rident_bytes(rec, players))
            r = int(rec['link']) >> 8
        rec = oracle.r_root(cfg)[0]
        got = [oracle.rident_bytes(rec, players)]
        for o in ords:
            rec = oracle.r_expand(cfg, rec)[o]
            got.append(oracle.rident_bytes(rec, players))
        assert got == want[::-1]
        if rank == 0:
            Path(out_file).write_text(json.dumps(dict(levels=len(sol.infos))))
    finally:
        dist.destroy_process_group()


def _run(world, case, worker=_worker):
    with tempfile.TemporaryDirectory() as d:
        init_file, out_file = os.path.join(d, 'init'), os.path.join(d, 'out')
        mp.spawn(worker, args=(world, init_file, case, out_file), nprocs=world, join=True)
        return json.loads(Path(out_file).read_text())


@pytest.mark.parametrize('world,case', [
    (2, (2, 6, None, 300, 16, 'const')),    # 2 players, unshuffled market, many rounds per level
    (3, (2, 10, 0, 500, 37, 'hash')),       # odd world size, shuffled market (seed 0), hash noise
    (3, (3, 8, 0, 400, 29, 'const')),       # 3 players
    (2, (4, 6, 3, 200, 13, 'const')),       # 4 players (the 7-bit-per-3-cards owner code)
])
def test_rsharded_matches_oracle(world, case):
    out = _run(world, case)
    assert out['max_rounds'] >= 3, out


def test_rsharded_keep_all_levels():
    """a beam wider than the early levels (every unique state is kept, no radix select) and narrower than the late ones"""
    out = _run(2, (2, 6, None, 3000, 1 << 20, 'const'))
    assert 0 < out['keep_all'] < out['levels'] - 1, out


def test_rsharded_rejects_other_policies():
    from rfake_backend import RFakeBackend
    from splendor_rl_gym_b200.sharded import Comm, RShardedSolver
    comm = Comm(torch.device('cpu'))
    cfg = _ocfg(2, 6, None)
    for kw in (dict(tie='det'), dict(identity='pyhash')):
        with pytest.raises(ValueError):
            RShardedSolver(RFakeBackend(cfg), comm, 100, **kw)
    be = RFakeBackend(cfg)
    be.noise = 'mt'
    with pytest.raises(ValueError):
        RShardedSolver(be, comm, 100)


def test_rsharded_turn_limit():
    """TURN_LIMIT (1000 in realistic mode) lowered to 6: same levels as the oracle up to and including level 6, then the
    search ends there with the line from the last queued state of level 6"""
    out = _run(2, (2, 15, 0, 300, 32, 6), _worker_turn_limit)
    assert out['levels'] == 7, out
