"""GPU tests (-m gpu) of realistic mode on the key-sharded driver: the spl_r* entry points of RCudaBackend (and, where the
row layer is shared, the speedrun rows of CudaBackend) against numpy and the CPU oracle on small hand-built inputs, RShardedSolver on one rank against oracle.RSolver level by level, and
MultiPlayerState.solve(shard=True) against the single-GPU search."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle
import splendor_rl_gym_b200 as S
from splendor_rl_gym_b200._lib import SplendorB200Error, lib
from splendor_rl_gym_b200.realistic import RConfig
from splendor_rl_gym_b200.sharded import Comm, CudaBackend, RCudaBackend, RShardedSolver

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def eng():
    return S.Engine.get(0)


def _cfgs(run, noise='const'):
    """(library config, oracle config) of a golden realistic run"""
    P, gpc, m = run['players'], run['gems_per_color'], run['market']
    cfg = RConfig(P, run['goal'], gpc, {'const': 0, 'hash': 1}[noise])
    for t, seq in enumerate((m['t1'], m['t2'], m['t3'])):
        cfg.deck_len[t] = len(seq)
        for i, c in enumerate(seq):
            cfg.deck[t][i] = c
    return cfg, oracle.make_rconfig(P, run['goal'], gpc, [m['t1'], m['t2'], m['t3']], noise)


def _run(golden, players, goal, seed, beam):
    return next(r for r in golden['realistic_runs'] if (r['players'], r['goal'], r['seed'], r['beam']) == (players, goal, seed, beam))


def _rows(recs, dev):
    return torch.from_numpy(np.ascontiguousarray(recs).view(np.int64).reshape(-1, 12).copy()).to(dev)


def _recs(rows):
    return rows.cpu().numpy().view(oracle.RREC_DTYPE).reshape(-1)


def _levels(ocfg, beam, upto):
    """queues 0..upto of the oracle's search"""
    s = oracle.RSolver(ocfg, beam)
    for _ in range(upto):
        s.step()
    out = [s.level(i) for i in range(upto + 1)]
    s.close()
    return out


@pytest.fixture(scope='module')
def sample(golden):
    """a 2-player search's queues 6..9 (distinct states) and a list with duplicates (each state of level 7 twice)"""
    run = _run(golden, 2, 15, 0, 2000)
    cfg, ocfg = _cfgs(run)
    lv = _levels(ocfg, run['beam'], 9)
    distinct = np.concatenate(lv[6:10])
    dup = np.concatenate([lv[7], lv[8][:50], lv[7]])
    return cfg, ocfg, lv, distinct, dup


# ------------------------------------------------------------------ ABI units
def test_rexpand_rows_links_with_rank_base(eng, sample):
    cfg, ocfg, lv, _, _ = sample
    be = RCudaBackend(eng, cfg)
    front = lv[5]
    base = 123_456
    got = _recs(be.expand_rows(_rows(front, eng.tdev), base))
    want = []
    for r, rec in enumerate(front):
        kids = oracle.r_expand(ocfg, rec)
        kids['link'] = [(base + r) << 8 | o for o in range(len(kids))]
        want.append(kids)
    assert got.tobytes() == np.concatenate(want).tobytes()
    # a capacity below the successor count reports the count
    out = torch.empty((4, 12), dtype=torch.int64, device=eng.tdev)
    m = C.c_int64()
    rc = lib.spl_rexpand_rows(eng._h, C.byref(cfg), _rows(front, eng.tdev).data_ptr(), len(front), 0, out.data_ptr(), 4,
                              C.byref(m), eng._stream())
    assert rc == -6 and m.value == len(got)


@pytest.fixture(scope='module')
def row_kinds(eng, sample):
    """per row kind of the key-sharded driver: (backend factory, queues 0..9 of a beam search as device rows, identity keys
    of device rows as host uint64 [n, KEY_COLS]).  The realistic queues are `sample`'s."""
    cfg, _, lv, _, _ = sample
    s = oracle.Solver(15, use_heuristic=True, heuristic_name='balanced', beam_width=2000)
    for _ in range(9):
        s.step()
    slv = []
    for i in range(10):
        st, lk = s.level(i)
        slv.append(torch.from_numpy(np.stack([st['lo'], st['hi'], st['aux'], lk], axis=1).view(np.int64).copy()).to(eng.tdev))
    return {
        'speedrun': (CudaBackend, slv, lambda rows: np.ascontiguousarray(rows[:, :2].cpu().numpy()).view(np.uint64)),
        'realistic': (lambda e: RCudaBackend(e, cfg), [_rows(q, eng.tdev) for q in lv], lambda rows: eng.rpack(cfg, _recs(rows))),
    }


# The row-layer tests below check each row kind: speedrun rows through CudaBackend (spl_route_keys, spl_dedup_flags,
# spl_compact_winners, spl_move_rows) and realistic rows through RCudaBackend (their spl_r* twins).
ROW_KINDS = ('speedrun', 'realistic')


@pytest.mark.parametrize('world', [1, 3, 8])
def test_rroute_keys_groups_counts_stability(eng, row_kinds, world):
    for kind in ROW_KINDS:
        _route_keys_groups_counts_stability(eng, row_kinds, kind, world)


def test_rdedup_flags_first_arrival_within_and_across_calls(eng, row_kinds):
    for kind in ROW_KINDS:
        _dedup_flags_first_arrival_within_and_across_calls(eng, row_kinds, kind)


def test_rcompact_winners_order_and_state_error(eng, row_kinds):
    for kind in ROW_KINDS:
        _compact_winners_order_and_state_error(eng, row_kinds, kind)


def test_rmove_rows_gather_scatter(eng, row_kinds):
    for kind in ROW_KINDS:
        _move_rows_gather_scatter(eng, row_kinds, kind)


def _route_keys_groups_counts_stability(eng, row_kinds, kind, world):
    make, lv, keys_of = row_kinds[kind]
    dup = torch.cat([lv[7], lv[8][:50], lv[7]])  # each state of level 7 twice
    send, counts = make(eng).route_keys(dup, world)
    keys = keys_of(dup)
    send = send.cpu().numpy().view(np.uint64)
    assert counts.sum() == len(dup) and len(send) == len(dup)
    if world == 1:
        assert (send == keys).all()
    # every key goes to one owner; inside a group the candidates keep their arrival order
    pos = {}
    for i, k in enumerate(keys):
        pos.setdefault(bytes(k), []).append(i)
    owner_of, start = {}, 0
    for g, c in enumerate(counts):
        prev = -1
        for k in send[start:start + c]:
            b = bytes(k)
            assert owner_of.setdefault(b, g) == g
            i = pos[b].pop(0)
            assert i > prev
            prev = i
        start += c
    assert all(not v for v in pos.values())
    if world == 8:  # the owner hash spreads the states
        assert counts.min() > 0.5 * len(dup) / world


def _dedup_flags_first_arrival_within_and_across_calls(eng, row_kinds, kind):
    make, lv, keys_of = row_kinds[kind]
    be = make(eng)
    be.reset_visited()
    dup = torch.cat([lv[7], lv[8][:50], lv[7]])
    keys = torch.from_numpy(keys_of(dup).view(np.int64).copy()).to(eng.tdev)
    f1 = be.dedup_flags(keys).cpu().numpy()
    seen, want = set(), []
    for k in keys.cpu().numpy():
        want.append(bytes(k) not in seen)
        seen.add(bytes(k))
    assert (f1 == np.array(want)).all()
    assert be.visited_count() == len(seen)
    # second call: states of the first lose, new ones win on their first arrival
    more = torch.cat([lv[8][40:80], lv[9][:30], lv[9][:30]])
    k2 = torch.from_numpy(keys_of(more).view(np.int64).copy()).to(eng.tdev)
    f2 = be.dedup_flags(k2).cpu().numpy()
    want2 = []
    for k in k2.cpu().numpy():
        want2.append(bytes(k) not in seen)
        seen.add(bytes(k))
    assert (f2 == np.array(want2)).all() and be.visited_count() == len(seen)
    be.reset_visited()
    assert be.visited_count() == 0 and be.dedup_flags(keys).cpu().numpy().sum() == len(set(bytes(k) for k in keys.cpu().numpy()))


def _compact_winners_order_and_state_error(eng, row_kinds, kind):
    make, lv, keys_of = row_kinds[kind]
    be = make(eng)
    cand = torch.cat(lv[6:10])  # distinct states
    send, counts = be.route_keys(cand, 3)
    keys = keys_of(cand)
    where = {bytes(k): i for i, k in enumerate(keys)}
    src = np.array([where[bytes(k)] for k in send.cpu().numpy().view(np.uint64)])
    rng = np.random.default_rng(0)
    flags = rng.integers(0, 2, len(cand)).astype(np.uint8)
    got = be.compact_winners(cand, torch.from_numpy(flags).to(eng.tdev))
    won = np.zeros(len(cand), bool)
    won[src[flags == 1]] = True
    assert got.cpu().numpy().tobytes() == cand.cpu().numpy()[won].tobytes()
    with pytest.raises(SplendorB200Error) as e:  # not the candidates of the last route
        be.compact_winners(cand[:-1], torch.from_numpy(flags[:-1]).to(eng.tdev))
    assert e.value.code == -7
    other_make, other_lv, _ = row_kinds[next(k for k in ROW_KINDS if k != kind)]
    n = min(len(cand), len(torch.cat(other_lv[6:10])))
    fresh = S.Engine(0, table_slots=1 << 12)
    try:
        with pytest.raises(SplendorB200Error) as e:  # no route on this context yet
            make(fresh).compact_winners(cand, torch.from_numpy(flags).to(eng.tdev))
        assert e.value.code == -7
        # the other row kind's route on as many candidates is not a route of this kind
        other_make(fresh).route_keys(torch.cat(other_lv[6:10])[:n], 3)
        with pytest.raises(SplendorB200Error) as e:
            make(fresh).compact_winners(cand[:n], torch.from_numpy(flags[:n]).to(eng.tdev))
        assert e.value.code == -7
    finally:
        fresh.close()


def _move_rows_gather_scatter(eng, row_kinds, kind):
    make, lv, _ = row_kinds[kind]
    be = make(eng)
    rows = torch.cat(lv[6:10])
    host = rows.cpu().numpy()
    perm = torch.from_numpy(np.random.default_rng(1).permutation(len(rows))).to(eng.tdev)
    g = be.move_rows(rows, perm, len(rows), False)
    assert g.cpu().numpy().tobytes() == host[perm.cpu().numpy()].tobytes()
    s = be.move_rows(g, perm, len(rows), True)
    assert s.cpu().numpy().tobytes() == host.tobytes()
    dst = torch.zeros_like(rows)
    be.scatter_into(dst, g, perm)
    assert dst.cpu().numpy().tobytes() == host.tobytes()


def test_rfirst_goal_vs_oracle_pts(eng, golden):
    run = _run(golden, 2, 6, None, 300)
    cfg, ocfg = _cfgs(run)
    s = oracle.RSolver(ocfg, run['beam'])
    s.run()
    be = RCudaBackend(eng, cfg)
    for lvl in (s.nlevels - 1, s.nlevels - 2, 3):
        recs = s.level(lvl)
        want = next((i for i, r in enumerate(recs) if oracle.r_pts(r, int(r['cur'])) >= run['goal']), -1)
        assert be.first_goal(_rows(recs, eng.tdev), run['goal']) == want
    assert be.first_goal(_rows(s.level(s.nlevels - 1), eng.tdev), run['goal']) == s.infos[-1]['goal_rank'] >= 0
    s.close()


# ------------------------------------------------------------------ the driver on one rank
def _check_driver(eng, cfg, ocfg, beam, block, what):
    sol = RShardedSolver(RCudaBackend(eng, cfg), Comm(eng.tdev), beam, block_parents=block)
    orc = oracle.RSolver(ocfg, beam)
    while True:
        gi, oi = sol.step(), orc.step()
        fields = ('frontier', 'goal_rank') if gi['ended'] else ('frontier', 'expanded', 'generated', 'unique', 'kept', 'goal_rank', 'visited')
        for f in fields:
            assert gi[f] == oi[f], (what, f, gi, oi)
        if gi['ended']:
            break
        assert _recs(sol.gather_frontier()).tobytes() == orc.level(oi['level'] + 1).tobytes(), (what, gi['level'])
    assert orc.done
    ranks, ords = sol.path()
    want = orc.path()
    assert len(ords) == len(want) - 1, what
    rec = oracle.r_root(ocfg)[0]
    for o, w in zip(ords, want[1:]):
        rec = oracle.r_expand(ocfg, rec)[o]
        assert oracle.rident_bytes(rec, ocfg.num_players) == oracle.rident_bytes(w, ocfg.num_players), what
    orc.close()
    return sol


@pytest.mark.parametrize('block', [1 << 22, 64])
def test_driver_one_rank_vs_oracle(eng, golden, block):
    """every golden realistic run, one round per level and (block 64) many rounds per level"""
    for run in golden['realistic_runs']:
        cfg, ocfg = _cfgs(run)
        what = f"p={run['players']} goal={run['goal']} seed={run['seed']} beam={run['beam']} block={block}"
        sol = _check_driver(eng, cfg, ocfg, run['beam'], block, what)
        assert len(sol.path()[1]) == run['plies'], what


def test_driver_beam_20000_known_answer(eng):
    """SURVEY.md 8c: 2 players, goal 15, market seed 0, beam 20 000 -> 53 plies, 977 184 expanded, 4 194 569 visited.
    Checked on the driver: every level against the oracle, the 53 plies of its line, and 977 184 expanded = its parents
    of all levels before the goal level + the goal's rank (the reference expands the states queued before the goal state
    in its last iteration; the driver stops at the goal).  The 4 194 569 visited include the states that partial last
    iteration inserts, which the driver never generates: that number is checked on the oracle, and the driver's visited
    count is checked against the oracle's up to the last level it expands."""
    m = S.CardMarket.from_full_deck(shuffle=True, seed=0)
    tiers = [list(m.tier1_visible + m.tier1_deck), list(m.tier2_visible + m.tier2_deck), list(m.tier3_visible + m.tier3_deck)]
    run = dict(players=2, goal=15, gems_per_color=4, market=dict(t1=tiers[0], t2=tiers[1], t3=tiers[2]))
    cfg, ocfg = _cfgs(run)
    sol = _check_driver(eng, cfg, ocfg, 20_000, 1 << 12, 'beam 20000')
    infos = sol.infos
    assert len(sol.path()[1]) == 53
    # the reference still expands the states queued before the goal state in its last iteration
    assert sum(i['expanded'] for i in infos[:-1]) + infos[-1]['goal_rank'] == 977_184
    s = oracle.RSolver(ocfg, 20_000)
    s.run()
    assert s.infos[-1]['visited'] == 4_194_569 and s.infos[-2]['visited'] == infos[-2]['visited']
    s.close()


def test_driver_hash_noise_vs_oracle(eng, golden):
    run = _run(golden, 3, 8, 0, 400)
    cfg, ocfg = _cfgs(run, 'hash')
    _check_driver(eng, cfg, ocfg, run['beam'], 50, 'noise=hash')


class _ZeroScores(RCudaBackend):
    """scores with negative values and both signed zeros, ties across -0.0 / +0.0 at the cut: every fourth state
    scores -0.0, the next +0.0, the rest (real score - 500)"""

    def score(self, heuristic, noise, rows, draws=None):
        s = super().score(heuristic, noise, rows, draws) - 500.0
        i = torch.arange(rows.shape[0], device=rows.device)
        s = torch.where(i % 4 == 0, torch.full_like(s, -0.0), s)
        s = torch.where(i % 4 == 1, torch.zeros_like(s), s)
        self.last = (rows.clone(), s.clone())
        return s


def test_cut_negative_scores_and_signed_zero(eng, golden):
    """from the third level on, half of the states score -0.0 or +0.0 and more than the beam of 1000 do: the cut falls
    inside that tie group and must split it by arrival order alone, as Python's stable sort does"""
    run = _run(golden, 2, 15, 0, 2000)
    cfg, _ = _cfgs(run)
    be = _ZeroScores(eng, cfg)
    beam = 1000
    sol = RShardedSolver(be, Comm(eng.tdev), beam, block_parents=128)
    cuts_in_zeros = 0
    for _ in range(7):
        info = sol.step()
        assert not info['ended']
        rows, sc = be.last
        sc = sc.cpu().numpy()
        order = sorted(range(len(sc)), key=lambda i: sc[i], reverse=True)[:beam]  # the reference's cut
        assert _recs(sol.gather_frontier()).tobytes() == _recs(rows)[order].tobytes(), info
        zeros = sc == 0
        if len(sc) > beam and sc[order[-1]] == 0:
            kept = np.zeros(len(sc), bool)
            kept[order] = True
            assert (sc < 0).any() and np.signbit(sc[zeros]).any() and (~np.signbit(sc[zeros])).any()
            assert (zeros & ~kept).any()  # the tie group straddles the cut
            cuts_in_zeros += 1
    assert cuts_in_zeros >= 3


def test_solve_shard_same_path_as_single_gpu(golden):
    for players, goal, seed, beam in ((2, 6, None, 300), (3, 8, 0, 400), (4, 6, 3, 200)):
        gpc = {2: 4, 3: 5, 4: 7}[players]
        cfg = S.GameConfig(num_players=players, target_points=goal, gems_per_color=gpc, infinite_resources=False)
        root = S.MultiPlayerState.newgame(cfg, shuffle_market=seed is not None, seed=seed)
        a = root.solve(beam_width=beam, verbose=False)
        stats = []
        b = root.solve(beam_width=beam, verbose=False, shard=True, stats=stats)
        assert [s.record().tobytes() for s in a] == [s.record().tobytes() for s in b]
        assert len(b) - 1 == _run(golden, players, goal, seed, beam)['plies'] and stats[-1]['ended'] == 1


def test_solve_shard_rejects_mt_noise():
    root = S.MultiPlayerState.newgame(S.GameConfig(num_players=2, target_points=6, gems_per_color=4, infinite_resources=False))
    with pytest.raises(ValueError):
        root.solve(beam_width=100, verbose=False, noise='mt', shard=True)


def test_context_usable_after_sharded_run(eng, golden):
    run = _run(golden, 2, 6, None, 300)
    cfg, ocfg = _cfgs(run)
    sol = RShardedSolver(RCudaBackend(eng, cfg), Comm(eng.tdev), run['beam'], block_parents=32)
    sol.run()
    root = oracle.r_root(ocfg)
    rs = eng.rsolver(cfg, root, run['beam'])
    rs.run()
    assert len(rs.path()[1]) == run['plies'] and [i['unique'] for i in rs.infos[:-1]] == [i['unique'] for i in sol.infos[:-1]]
    rs.close()
    sp = eng.solver(0, 0, 6, True, 'balanced', 300)
    orc = oracle.Solver(6, use_heuristic=True, heuristic_name='balanced', beam_width=300)
    sp.run()
    orc.run()
    assert [i['unique'] for i in sp.infos[:-1]] == [i['unique'] for i in orc.infos[:-1]]
    sp.close()



def _gloo_worker(rank, world, init_file, case, out_file):
    """one rank of a gloo process group on cuda:0: the real RCudaBackend, with the collectives staged through the host"""
    import torch.distributed as dist
    dist.init_process_group('gloo', init_method=f'file://{init_file}', rank=rank, world_size=world)
    try:
        players, goal, seed, beam, block = case
        eng = S.Engine(0)
        comm = Comm(eng.tdev)
        assert comm.stage and comm.world == world
        m = S.CardMarket.from_full_deck(shuffle=seed is not None, seed=seed)
        tiers = [list(m.tier1_visible + m.tier1_deck), list(m.tier2_visible + m.tier2_deck), list(m.tier3_visible + m.tier3_deck)]
        run = dict(players=players, goal=goal, gems_per_color={2: 4, 3: 5, 4: 7}[players], market=dict(t1=tiers[0], t2=tiers[1], t3=tiers[2]))
        cfg, ocfg = _cfgs(run)
        sol = RShardedSolver(RCudaBackend(eng, cfg), comm, beam, block_parents=block)
        orc = oracle.RSolver(ocfg, beam)
        rounds = 0
        while True:
            gi, oi = sol.step(), orc.step()
            fields = ('frontier', 'goal_rank') if gi['ended'] else ('frontier', 'expanded', 'generated', 'unique', 'kept', 'goal_rank', 'visited')
            for f in fields:
                assert gi[f] == oi[f], (rank, f, gi, oi)
            rounds = max(rounds, -(-(-(-gi['frontier'] // block)) // world))
            if gi['ended']:
                break
            assert _recs(sol.gather_frontier()).tobytes() == orc.level(oi['level'] + 1).tobytes(), (rank, gi['level'])
        ranks, ords = sol.path()
        want = orc.path()
        rec = oracle.r_root(ocfg)[0]
        for o, w in zip(ords, want[1:]):
            rec = oracle.r_expand(ocfg, rec)[o]
            assert oracle.rident_bytes(rec, players) == oracle.rident_bytes(w, players)
        assert len(ords) == len(want) - 1
        visited = [int(x) for x in comm.gather_ints(sol.b.visited_count())[:, 0]]
        if rank == 0:
            import json
            from pathlib import Path
            Path(out_file).write_text(json.dumps(dict(rounds=rounds, visited=visited)))
        orc.close()
        eng.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('world,case', [
    (2, (2, 15, 0, 2000, 128)),    # 2 players, seed 0, many rounds per level
    (3, (3, 8, 0, 400, 29)),       # odd world size, 3 players
    (4, (4, 6, 3, 200, 16)),       # 4 players
])
def test_driver_several_ranks_on_one_gpu_vs_oracle(world, case):
    """world 2-4 over gloo on one GPU: the device side of every collective (6-word keys out, winner bytes back, the
    distributed radix select, count_less ranks, redistribution of 96-byte rows) with the real kernels, every level
    against the oracle; each rank's visited table holds a share of the states"""
    import json
    import os
    import tempfile
    from pathlib import Path

    import torch.multiprocessing as mp
    with tempfile.TemporaryDirectory() as d:
        init_file, out_file = os.path.join(d, 'init'), os.path.join(d, 'out')
        mp.spawn(_gloo_worker, args=(world, init_file, case, out_file), nprocs=world, join=True)
        out = json.loads(Path(out_file).read_text())
    assert out['rounds'] >= 3 and len(out['visited']) == world
    assert min(out['visited']) > 0.5 * sum(out['visited']) / world, out
