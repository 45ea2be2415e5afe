"""GPU tests (-m gpu) of the speedrun sharded drivers with 2 to 8 ranks sharing one GPU.

Every case spawns `world` processes in a gloo process group on cuda:0: each rank runs the real kernels on its own Engine,
and Comm stages the collectives through host memory.  Rank 0 steps the CPU oracle beside the driver and compares every
level (counters, queue bytes: key, aux, link) and, at the end, the line.  Covered: the card-set-sharded driver
(GroupedShardedSolver: buy records stored into the peers' receive buffers over CUDA IPC or sent by all-to-all, merged
score dictionaries, threshold ties split across ranks, sample-sort ranks), the key-sharded driver (ShardedSolver +
CudaBackend), and State.solve under a process group, including its fallback after a score-dictionary overflow.  At world 1
the sample-sort primitives spl_gs_rank_sort and spl_gs_partition are checked against numpy."""
import ctypes as C
import json
import os
import random
import tempfile
import zlib
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import oracle
import splendor_rl_gym_b200 as S
from splendor_rl_gym_b200._lib import lib
from splendor_rl_gym_b200.sharded import Comm, CudaBackend, DictionaryOverflow, GroupedShardedSolver, ShardedSolver

pytestmark = pytest.mark.gpu

SPL_E_INVALID = -1
FIELDS = ('frontier', 'generated', 'unique', 'kept', 'goal_rank', 'visited')
GOLDEN = Path(__file__).parent / 'golden'
# (heuristic, beam, goal) whose grouped search meets a level with more distinct scores than the score dictionary holds
# (2048): level 22, on any number of ranks, since the merged dictionary is that of the whole level
OVERFLOW, OVERFLOW_LEVEL = ('balanced', 40_000, 40), 22


# ------------------------------------------------------------------ process groups on one GPU
def _entry(rank, world, init_file, out_file, fn, args):
    """one rank: gloo group, its own Engine on cuda:0; fn(eng, comm, *args) -> result, written as JSON by rank 0"""
    dist.init_process_group('gloo', init_method=f'file://{init_file}', rank=rank, world_size=world)
    try:
        eng = S.Engine(0)
        comm = Comm(eng.tdev)
        assert comm.stage and comm.world == world and comm.rank == rank
        out = fn(eng, comm, *args)
        peer = getattr(eng, '_peer_recv', None)
        if peer is not None:
            peer.release()  # collective: every mapping is closed before its owner frees the buffer
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


def _oracle_line(orc):
    """(ranks, ordinals) of the oracle's line: back from the goal state, or from the last state dequeued when the queue
    ran out, through the per-level links"""
    last = len(orc.infos) - 1
    r = orc.infos[-1]['goal_rank']
    if r < 0:
        r = len(orc.level(last)[0]) - 1
    ranks, ords = [0] * (last + 1), [0] * last
    for lv in range(last, 0, -1):
        ranks[lv] = r
        link = int(orc.level(lv)[1][r])
        ords[lv - 1], r = link & 0xff, link >> 8
    ranks[0] = r
    return ranks, ords


def _step_vs_oracle(sol, orc, what):
    """step the driver (every rank) and the oracle (rank 0 only: orc is None elsewhere) until the search ends, comparing
    every level; every rank gathers the queue and walks the line, since both are collective.  -> the driver's infos"""
    while True:
        gi = sol.step()
        if orc is not None:
            oi = orc.step()
            # at the goal the reference still expands the states queued before the goal state; the drivers skip that work
            fields = ('frontier', 'goal_rank') if gi['ended'] and gi['goal_rank'] >= 0 else FIELDS
            assert {f: gi[f] for f in fields} == {f: oi[f] for f in fields}, (what, gi, oi)
            assert bool(gi['ended']) == orc.done, (what, gi['level'])
        if gi['ended']:
            break
        fr = sol.gather_frontier().cpu().numpy().view(np.uint64)
        if orc is not None:
            st, lk = orc.level(oi['level'] + 1)
            assert fr.tobytes() == np.stack([st['lo'], st['hi'], st['aux'], lk], 1).tobytes(), (what, gi['level'])
    ranks, ords = sol.path()
    if orc is not None:
        assert (list(ranks), list(ords)) == _oracle_line(orc), what
    return sol.infos


# ------------------------------------------------------------------ card-set-sharded driver
def _grouped(eng, comm, hname, beam, rounds, peer, goal=15):
    """one GroupedShardedSolver search against the oracle -> per-level coverage: tie splits, rounds, unique states per rank"""
    if not peer:
        os.environ['SPL_NO_P2P'] = '1'
    what = f'grouped {hname} beam={beam} goal={goal} rounds={rounds} world={comm.world} peer={peer}'
    sol = GroupedShardedSolver(eng, comm, 0, 0, goal, hname, beam, 'const', round_parents=rounds)
    orc = oracle.Solver(goal, use_heuristic=True, heuristic_name=hname, beam_width=beam) if comm.rank == 0 else None
    try:
        assert (sol.peer is not None) == peer, what
        infos = _step_vs_oracle(sol, orc, what)
        expanded = [i for i in infos if 'local_unique' in i]
        local = comm.gather_ints(*[i['local_unique'] for i in expanded])  # [rank, level]
    finally:
        sol.close()
        if orc is not None:
            orc.close()
    return dict(levels=len(infos), tie_split=[i['tie_split'] for i in expanded if 'tie_split' in i],
                rounds=[-(-i['frontier'] // rounds) for i in expanded], local_unique=local.tolist(),
                goal_rank=sol.goal_rank, last=infos[-1])


@pytest.mark.parametrize('world,hname,beam,rounds,peer', [
    (2, 'aggressive', 20_000, 1 << 27, True),   # buy records stored into the other process's receive buffer (CUDA IPC)
    (2, 'aggressive', 20_000, 1 << 27, False),  # SPL_NO_P2P=1: send buffer and all-to-all
    (3, 'simple', 50_000, 3000, True),          # odd world, many rounds, mass score ties split across ranks
    (4, 'balanced', 5_000, 1024, True),         # window edges, 4-way sample sort
    (8, 'aggressive', 2_000, 1 << 27, True),    # early levels where most ranks own no state (k_local = 0 in the sample sort)
])
def test_grouped_driver_several_ranks_vs_oracle(world, hname, beam, rounds, peer):
    out = _spawn(world, _grouped, hname, beam, rounds, peer)
    local = np.array(out['local_unique'])
    assert out['last']['ended'] and out['last']['goal_rank'] >= 0, out['last']
    assert (local.max(axis=1) > 0).all(), local  # every rank owns states at some level
    if hname == 'simple':
        assert any(out['tie_split']), out['tie_split']
    if rounds < 1 << 27:
        assert max(out['rounds']) >= 2, out['rounds']
    if world == 8:
        assert (local == 0).any(), local


def _grouped_runs_out(eng, comm):
    return [_grouped(eng, comm, hname, beam, 1 << 27, True, goal=255)
            for hname in ('simple', 'balanced', 'aggressive', 'efficiency') for beam in (1, 2, 5)]


def test_grouped_driver_several_ranks_runs_out_of_states():
    """beams 1, 2 and 5 to goal 255 on 3 ranks: the queue runs out after 110-163 levels, and the line starts from the
    last state dequeued, rank N - 1 of the last queue"""
    for out in _spawn(3, _grouped_runs_out):
        last = out['last']
        assert out['levels'] > 100 and last['ended'] and last['kept'] == 0 and last['goal_rank'] == -1, last
        assert out['goal_rank'] == last['frontier'] - 1, out
        assert (np.array(out['local_unique']).max(axis=1) > 0).all()


# ------------------------------------------------------------------ key-sharded driver with the real kernels
def _key_sharded(eng, comm, cases):
    out = []
    for goal, use_h, hname, beam, tie, noise, block, identity in cases:
        what = f'key-sharded {hname if use_h else "bfs"} beam={beam} {tie}/{noise} goal={goal} block={block} {identity} world={comm.world}'
        sol = ShardedSolver(CudaBackend(eng), comm, 0, 0, goal, use_h, hname, beam, tie, noise, block_parents=block,
                            identity=identity)
        orc = None
        if comm.rank == 0:
            orc = oracle.Solver(goal, use_heuristic=use_h, heuristic_name=hname, beam_width=beam, policy=tie, noise=noise,
                                identity=identity)
        try:
            infos = _step_vs_oracle(sol, orc, what)
        finally:
            if orc is not None:
                orc.close()
        expanded = [i for i in infos if not i['ended']]
        out.append(dict(what=what, block=block, use_h=use_h,
                        rounds=max(-(-(-(-i['frontier'] // block)) // comm.world) for i in expanded),
                        cut=any(i['unique'] > i['kept'] for i in expanded),
                        visited=comm.gather_ints(eng.visited_count())[:, 0].tolist()))
    return out


KEY_CASES = {
    2: [(4, False, 'simple', 0, 'stable', 'const', 64, 'key'),            # exhaustive BFS, many rounds of 64-parent blocks
        (6, True, 'balanced', 300, 'stable', 'const', 37, 'key'),         # arrival-order ties over multi-round arrival indices
        (6, True, 'aggressive', 257, 'det', 'hash', 50, 'key'),           # key tie-break: the key threshold words across ranks
        (15, True, 'efficiency', 7, 'stable', 'hash', 3, 'key'),          # tiny beam, ragged 3-parent blocks
        (6, True, 'balanced', 300, 'stable', 'const', 37, 'pyhash'),      # visited set keyed by the reference's State.hash
        (4, False, 'simple', 0, 'stable', 'const', 64, 'pyhash'),         # ... exhaustive BFS
        (15, True, 'balanced', 20_000, 'det', 'hash', 4096, 'key')],      # wide beam, several rounds per level
    3: [(4, False, 'simple', 0, 'stable', 'const', 1000, 'key'),          # odd world size, ragged last block
        (6, True, 'simple', 100, 'stable', 'const', 16, 'key'),           # mass ties (simple with const noise)
        (6, True, 'balanced', 300, 'stable', 'const', 1 << 20, 'key')],   # one round per level
}


@pytest.mark.parametrize('world', sorted(KEY_CASES))
def test_key_sharded_driver_several_ranks_vs_oracle(world):
    for case in _spawn(world, _key_sharded, KEY_CASES[world]):
        assert min(case['visited']) > 0, case  # every rank's visited table holds a share of the states
        if case['use_h']:
            assert case['cut'], case  # some level holds more states than the beam
        if case['block'] < 1 << 20:
            assert case['rounds'] >= 2, case


# ------------------------------------------------------------------ State.solve under a process group
def _line_key(line):
    return [(s.cards, s.bonus, s.gems, s.pts, s.saved) for s in line]


def _oracle_line_key(orc):
    return [tuple(oracle.unpack_state(w)[f] for f in ('cards', 'bonus', 'gems', 'pts', 'saved')) for w in orc.path()]


def _solve(eng, comm):
    """State.solve as torchrun users call it, with the drivers' step() counted (and the grouped driver's overflow seen)"""
    calls = dict(grouped=0, key=0, overflow=[])
    g_step, k_step = GroupedShardedSolver.step, ShardedSolver.step

    def grouped_step(self):
        calls['grouped'] += 1
        try:
            return g_step(self)
        except DictionaryOverflow:
            calls['overflow'].append(self.level)
            raise

    def key_step(self):
        calls['key'] += 1
        return k_step(self)

    GroupedShardedSolver.step, ShardedSolver.step = grouped_step, key_step
    out = {}
    try:
        for name, (hname, beam, goal) in (('grouped', ('aggressive', 20_000, 15)), ('overflow', OVERFLOW)):
            for k in ('grouped', 'key'):
                calls[k] = 0
            calls['overflow'] = []
            line = S.State.newgame().solve(goal, use_heuristic=True, heuristic_name=hname, beam_width=beam, verbose=False,
                                           engine=eng)
            if comm.rank == 0:
                orc = oracle.Solver(goal, use_heuristic=True, heuristic_name=hname, beam_width=beam)
                orc.run()
                assert _line_key(line) == _oracle_line_key(orc), name
                orc.close()
            digest = zlib.crc32(repr(_line_key(line)).encode())
            out[name] = dict(lines=comm.gather_ints(len(line), digest).tolist(), grouped=calls['grouped'], key=calls['key'],
                             overflow=comm.gather_ints(*(calls['overflow'] or [-1]))[:, 0].tolist())
        calls['key'] = 0
        runs = [r for r in json.loads((GOLDEN / 'mt_runs.json').read_text()) if r['mode'] == 'speedrun']
        for run in runs:
            what = f"mt {run['heuristic']} goal={run['goal']} beam={run['beam']} seed={run['seed']} rank={comm.rank}"
            random.seed(run['seed'])
            line = S.State.newgame().solve(goal_pts=run['goal'], use_heuristic=True, heuristic_name=run['heuristic'],
                                           beam_width=run['beam'], verbose=False, noise='mt', engine=eng)
            assert [repr(s) for s in line] == [p['repr'] for p in run['path']], what
            assert [(s.saved, s.pts) for s in line] == [(p['saved'], p['pts']) for p in run['path']], what
            # every rank leaves the global generator where the reference leaves it
            assert [random.randint(1, 100) for _ in range(4)] == run['after'], what
        out['mt'] = dict(runs=len(runs), key=calls['key'])
    finally:
        GroupedShardedSolver.step, ShardedSolver.step = g_step, k_step
    return out


def test_state_solve_two_ranks():
    """stable / const runs on the card-set-sharded driver; a level with more distinct scores than the score dictionary
    makes every rank rerun the search on the key-sharded driver; noise 'mt' runs on the key-sharded driver and leaves
    every rank's `random` where the reference leaves it"""
    out = _spawn(2, _solve)
    g, o = out['grouped'], out['overflow']
    for case in (g, o):
        assert len({tuple(x) for x in case['lines']}) == 1, case  # every rank returns the same line
    assert g['grouped'] > 10 and g['key'] == 0 and g['overflow'] == [-1, -1], g
    assert o['overflow'] == [OVERFLOW_LEVEL, OVERFLOW_LEVEL], o  # both ranks overflow at the same level
    assert o['grouped'] == o['overflow'][0] + 1 and o['key'] > o['overflow'][0], o
    assert out['mt']['runs'] == 5 and out['mt']['key'] > 5 * 10, out['mt']


# ------------------------------------------------------------------ sample-sort primitives at world 1
@pytest.fixture(scope='module')
def eng():
    return S.Engine.get(0)


@pytest.fixture
def gs(eng):
    sol = GroupedShardedSolver(eng, Comm(eng.tdev), 0, 0, 15, 'aggressive', 20_000, 'const')
    yield sol
    sol.close()


def _rank_sort(sol, y, y_bits, base):
    """spl_gs_rank_sort of host words y -> host ranks"""
    n = len(y)
    dy = torch.from_numpy(y.view(np.int64)).to(sol.eng.tdev) if n else None
    out = torch.full((max(n, 1),), -7, dtype=torch.int64, device=sol.eng.tdev)
    rc = lib.spl_gs_rank_sort(sol._h, dy.data_ptr() if n else None, n, y_bits, base, out.data_ptr(), sol._st())
    assert rc == 0, (n, y_bits, rc)
    return out.cpu().numpy()


def _want_ranks(y, base):
    want = np.empty(len(y), np.int64)
    want[np.argsort(y, kind='stable')] = base + np.arange(len(y))
    return want


def _distinct_words(rng, n, y_bits):
    if n > (1 << y_bits) // 4:
        return np.sort(rng.choice(1 << y_bits, n, replace=False).astype(np.uint64))
    y = np.unique(rng.integers(0, 1 << y_bits, n + n // 8 + 8, dtype=np.uint64))
    return np.sort(rng.permutation(y)[:n])


def test_rank_sort_vs_numpy(gs):
    """ranks_out[i] = base + rank of word i among the words, at the one-sweep digit edges (10-bit digits: y_bits 10, 11, 20,
    21, 30, 31, 53) and sort-tile edges (4096 words), for sorted, reversed and shuffled input"""
    rng = np.random.default_rng(11)
    bases = (0, 12_345, (1 << 33) + 7)
    checked = 0
    for y_bits in (10, 11, 20, 21, 30, 31, 53):
        for n in (0, 1, 2, 4095, 4096, 4097, 12_289, 1_048_579):
            if n > 1 << y_bits:
                continue
            y = _distinct_words(rng, n, y_bits)
            for i, order in enumerate((y, y[::-1].copy(), rng.permutation(y))):
                base = bases[(i + n) % 3]
                got = _rank_sort(gs, order, y_bits, base)
                if n:
                    assert (got == _want_ranks(order, base)).all(), (y_bits, n, i, base)
                else:
                    assert (got == -7).all()  # n = 0 leaves the output untouched
                checked += 1
    assert checked == 3 * (3 + 3 + 7 + 8 + 8 + 8 + 8)


def test_rank_sort_rejects_too_many_words(gs):
    """2^30 words is over the per-rank limit: refused before any device work (the word pointer is never read)"""
    out = torch.empty(1, dtype=torch.int64, device=gs.eng.tdev)
    assert lib.spl_gs_rank_sort(gs._h, None, 1 << 30, 40, 0, out.data_ptr(), gs._st()) == SPL_E_INVALID


def test_partition_and_rank_sort_on_real_survivors(gs):
    """spl_gs_partition against np.searchsorted(side='left') on the sorted survivors of every level of a search (captured
    where the driver computes their global ranks), and spl_gs_rank_sort of the same words shuffled"""
    rng = np.random.default_rng(12)
    seen = []
    global_ranks = gs._global_ranks

    def check(y_ptr, k_local, y_bits, k_total):
        y = gs._dev(y_ptr, (k_local,)).cpu().numpy().view(np.uint64) if k_local else np.zeros(0, np.uint64)
        assert (y[1:] > y[:-1]).all() and (y >> np.uint64(y_bits) == 0).all()  # ascending, distinct, y_bits wide
        top = np.uint64((1 << 64) - 1)
        lo, hi = (int(y[0]), int(y[-1])) if k_local else (1, 1)
        probes = [0, max(lo - 1, 0), lo, lo + 1, hi - 1, hi, hi + 1, int(top), lo, lo, hi, hi]
        probes += [int(v) for v in rng.choice(y, 24)] if k_local else [5] * 24                   # equal to words
        probes += [int(v) + 1 for v in rng.choice(y, 20)] if k_local else [7] * 20               # just above words
        probes += [int(v) for v in rng.integers(lo, hi + 1, 8, dtype=np.uint64)]                 # anywhere between
        probes = np.sort(np.array(probes, dtype=np.uint64))
        assert len(probes) == 64
        bounds = (C.c_int64 * 65)(*([-3] * 65))
        rc = lib.spl_gs_partition(gs._h, (C.c_uint64 * 64)(*probes.tolist()), 64, bounds, gs._st())
        assert rc == 0
        assert (np.array(bounds[:64]) == np.searchsorted(y, probes, side='left')).all(), y_bits
        assert lib.spl_gs_partition(gs._h, (C.c_uint64 * 65)(*probes.tolist(), 0), 65, bounds, gs._st()) == SPL_E_INVALID
        assert lib.spl_gs_partition(gs._h, None, 0, None, gs._st()) == 0
        assert bounds[64] == -3
        if k_local:
            shuffled = rng.permutation(y)
            assert (_rank_sort(gs, shuffled, y_bits, 99) == _want_ranks(shuffled, 99)).all(), y_bits
        seen.append((k_local, y_bits))
        return global_ranks(y_ptr, k_local, y_bits, k_total)

    gs._global_ranks = check
    while not gs.step()['ended']:
        pass
    assert len(seen) > 10 and max(k for k, _ in seen) == 20_000
