"""Batched realistic search (spl_rbatch_*, solve_many) against the same games solved one by one (spl_rsolver), on one GPU.

Workloads: 2 players to 15 points, market seeds 0..B-1, beam 20 000 (the reference's default width), B in --sizes; and
one mixed batch of 2- and 3-player games (even seeds 2 players, odd seeds 3 players, 15 points).  After one untimed
warm-up of each path, every workload is timed --reps times per path, the two paths alternating (batch first, then
sequential first), with a host clock around work that ends in a device synchronise.  Reported per workload:
  solver level:   games/s and expanded states/s of both paths (best rep), the batch's per-level phase split summed over
                  its levels (count = goal test + count, expand, probe = dedup + winners, score, cut = segmented cut)
  end to end:     solve_many (line building included) and the loop of MultiPlayerState.solve(), once each
  parity:         every game's (plies, visited, line digest) equal between the two end-to-end paths
One JSON line per workload (and a header line with the GPU's name and power limit) to stdout and to --out.

    python tools/rbatch_bench.py --out profiles/rb1_rbatch_bench.jsonl
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_header():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return {'gpu': q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None}


def roots_for(S, kind, B):
    out = []
    for seed in range(B):
        p = 3 if kind == 'mixed' and seed % 2 else 2
        cfg = S.GameConfig(num_players=p, target_points=15, gems_per_color={2: 4, 3: 5}[p], infinite_resources=False)
        out.append(S.MultiPlayerState.newgame(cfg, shuffle_market=True, seed=seed))
    return out


def run_batch(eng, roots, beam):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    sol = eng.rbatch_solver([r.rconfig() for r in roots], __import__('numpy').concatenate([r.record() for r in roots]),
                            [beam] * len(roots), keep_links=False)
    infos = sol.run()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    sol.close()
    ph = {k: sum(i[f] for i in infos) for k, f in (('count', 'ms_count'), ('expand', 'ms_expand'), ('probe', 'ms_resolve'),
                                                   ('score', 'ms_select'), ('cut', 'ms_sort'))}
    return dt, sum(i['expanded'] for i in infos), len(infos), ph


def run_sequential(eng, roots, beam):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    expanded = 0
    for r in roots:
        sol = eng.rsolver(r.rconfig(), r.record(), beam, keep_links=False)
        expanded += sum(i['expanded'] for i in sol.run())
        sol.close()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, expanded


def digest(line):
    h = hashlib.sha256()
    for s in line:
        r = s.record()[0]
        h.update(r['p'][:s.config.num_players].tobytes() + r['vis'].tobytes() + bytes([s.current_player]))
    return h.hexdigest()[:16]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--sizes', default='1,16,64,128')
    ap.add_argument('--mixed', type=int, default=32, help='games of the mixed 2/3-player batch (0: none)')
    ap.add_argument('--beam', type=int, default=20_000)
    ap.add_argument('--reps', type=int, default=2)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    import torch

    import splendor_rl_gym_b200 as S
    eng = S.Engine.get(0)
    lines_out = [dict(gpu_header(), torch_device=torch.cuda.get_device_name(0), beam=a.beam, reps=a.reps)]
    print(json.dumps(lines_out[0]), flush=True)
    warm = roots_for(S, '2p', 4)
    run_batch(eng, warm, a.beam)
    run_sequential(eng, warm[:1], a.beam)
    work = [('2p', int(b)) for b in a.sizes.split(',') if b] + ([('mixed', a.mixed)] if a.mixed else [])
    for kind, B in work:
        roots = roots_for(S, kind, B)
        tb, ts = [], []
        for rep in range(a.reps):
            order = ('batch', 'seq') if rep % 2 == 0 else ('seq', 'batch')
            for which in order:
                if which == 'batch':
                    dt, exp_b, levels, ph = run_batch(eng, roots, a.beam)
                    tb.append(dt)
                else:
                    dt, exp_s = run_sequential(eng, roots, a.beam)
                    ts.append(dt)
        # end to end, with the parity check of every game
        st_b = []
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        many = S.solve_many(roots, beam_width=a.beam, engine=eng, stats=st_b)
        e2e_b = time.perf_counter() - t0
        t0 = time.perf_counter()
        seq, seq_visited = [], []
        for r in roots:
            st = []
            seq.append(r.solve(beam_width=a.beam, verbose=False, engine=eng, stats=st))
            seq_visited.append(st[-1]['visited'])
        e2e_s = time.perf_counter() - t0
        batch_visited = [next(lv['games'][g]['visited'] for lv in reversed(st_b) if lv['games'][g]['ended'])
                         for g in range(B)]
        same = all((len(m), v, digest(m)) == (len(s_), w, digest(s_))
                   for m, s_, v, w in zip(many, seq, batch_visited, seq_visited))
        rec = dict(workload=kind, games=B, beam=a.beam, levels=levels,
                   batch_s=min(tb), seq_s=min(ts), batch_s_all=tb, seq_s_all=ts,
                   batch_games_per_s=B / min(tb), seq_games_per_s=B / min(ts), speedup=min(ts) / min(tb),
                   batch_expanded_per_s=exp_b / min(tb), seq_expanded_per_s=exp_s / min(ts),
                   batch_phase_ms=ph, e2e_solve_many_s=e2e_b, e2e_sequential_solve_s=e2e_s,
                   plies=[len(m) - 1 for m in many], parity=same)
        lines_out.append(rec)
        print(json.dumps(rec), flush=True)
        if not same:
            print('PARITY MISMATCH between solve_many and solve()', file=sys.stderr)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            for r in lines_out:
                f.write(json.dumps(r) + '\n')
    return 0 if all(r.get('parity', True) for r in lines_out) else 1


if __name__ == '__main__':
    sys.exit(main())
