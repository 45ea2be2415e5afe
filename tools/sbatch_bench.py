"""Batched speedrun search (spl_sbatch_*, State.solve_many) against the same games solved one by one (spl_solver), on
one GPU.

Workloads:
  sweep  the four heuristics x beams {1 000, 20 000, 300 000} x goals {10, 15} from State.newgame() (24 games): the
         comparison of heuristics across widths and goals that speedrun users run
  mid    64 mid-game roots (seeded walks of 4..11 plies from the new game), goal 15, the four heuristics in turn, beam
         300 000 (the reference's default width): the fastest win from many positions
  one    a batch of one: aggressive, goal 15, beam 300 000
After one untimed warm-up of each path, every workload is timed --reps times per path, the two paths alternating
(batch first, then sequential first), with a host clock around work that ends in a device synchronise.  The sequential
path is what State.solve() runs: the card-set-grouped level for beam search.  Reported per workload:
  solver level:   games/s and expanded states/s of both paths (best rep), the batch's per-level phase split summed over
                  its levels (count = goal test + count, expand, probe = dedup + winners, score, cut = key passes and
                  segmented cut)
  end to end:     State.solve_many (lines included) and the loop of State.solve(), once each: times, games/s and
                  expanded states/s
  parity:         every game's (moves, visited, line digest) equal between the two end-to-end paths
One JSON line per workload (and a header line with the GPU's name and power limit) to stdout and to --out.

    python tools/sbatch_bench.py --out profiles/sb1_sbatch_bench.jsonl
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

HEURISTICS = ('simple', 'balanced', 'aggressive', 'efficiency')
M64 = (1 << 64) - 1


def gpu_header():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return {'gpu': q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None}


def workload(S, kind):
    """[(root, goal, heuristic, beam)]"""
    new = S.State.newgame()
    if kind == 'sweep':
        return [(new, goal, h, beam) for goal in (10, 15) for beam in (1000, 20_000, 300_000) for h in HEURISTICS]
    if kind == 'one':
        return [(new, 15, 'aggressive', 300_000)]
    games = []
    for i in range(64):
        s = new
        for ply in range(4 + i % 8):
            succ = list(s)
            s = succ[(i * 7 + ply * 13) % len(succ)]
        games.append((s, 15, HEURISTICS[i % 4], 300_000))
    return games


def run_batch(eng, games):
    import numpy as np
    import torch
    rows = np.array([(k & M64, k >> 64, a, M64) for k, a in (r.record() for r, *_ in games)], dtype=np.uint64)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    sol = eng.sbatch_solver(rows, [g for _, g, _, _ in games], [True] * len(games), [h for _, _, h, _ in games],
                            [b for *_, b in games], keep_links=False)
    infos = sol.run()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    sol.close()
    ph = {k: sum(i[f] for i in infos) for k, f in (('count', 'ms_count'), ('expand', 'ms_expand'), ('probe', 'ms_resolve'),
                                                   ('score', 'ms_select'), ('cut', 'ms_sort'))}
    return dt, sum(i['expanded'] for i in infos), len(infos), ph


def run_sequential(eng, games):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    expanded = 0
    for root, goal, h, beam in games:
        k, a = root.record()
        sol = eng.solver(k, a, goal, True, h, beam, keep_links=False)
        expanded += sum(i['expanded'] for i in sol.run())
        sol.close()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, expanded


def digest(line):
    return hashlib.sha256(repr([(s.cards, s.bonus, s.gems, s.pts, s.saved) for s in line]).encode()).hexdigest()[:16]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--workloads', default='sweep,mid,one')
    ap.add_argument('--reps', type=int, default=2)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    import torch

    import splendor_rl_gym_b200 as S
    eng = S.Engine.get(0)
    lines_out = [dict(gpu_header(), torch_device=torch.cuda.get_device_name(0), reps=a.reps)]
    print(json.dumps(lines_out[0]), flush=True)
    warm = [(S.State.newgame(), 10, h, 1000) for h in HEURISTICS]
    run_batch(eng, warm)
    run_sequential(eng, warm[:1])
    for kind in a.workloads.split(','):
        games = workload(S, kind)
        B = len(games)
        tb, ts = [], []
        for rep in range(a.reps):
            for which in (('batch', 'seq') if rep % 2 == 0 else ('seq', 'batch')):
                if which == 'batch':
                    dt, exp_b, levels, ph = run_batch(eng, games)
                    tb.append(dt)
                else:
                    dt, exp_s = run_sequential(eng, games)
                    ts.append(dt)
        # end to end, with the parity check of every game
        roots, goals, names, beams = (list(x) for x in zip(*games))
        st_b = []
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        many = S.State.solve_many(roots, goals, use_heuristic=True, heuristic_name=names, beam_width=beams, engine=eng, stats=st_b)
        e2e_b = time.perf_counter() - t0
        t0 = time.perf_counter()
        seq, seq_visited, exp_e2e_s = [], [], 0
        for root, goal, h, beam in games:
            st = []
            seq.append(root.solve(goal, use_heuristic=True, heuristic_name=h, beam_width=beam, verbose=False, engine=eng, stats=st))
            seq_visited.append(st[-1]['visited'])
            exp_e2e_s += sum(i['expanded'] for i in st)
        e2e_s = time.perf_counter() - t0
        exp_e2e_b = sum(i['expanded'] for i in st_b)
        batch_visited = [next(lv['games'][g]['visited'] for lv in reversed(st_b) if lv['games'][g]['ended']) for g in range(B)]
        same = all((len(m), v, digest(m)) == (len(s_), w, digest(s_))
                   for m, s_, v, w in zip(many, seq, batch_visited, seq_visited))
        rec = dict(workload=kind, games=B, levels=levels,
                   batch_s=min(tb), seq_s=min(ts), batch_s_all=tb, seq_s_all=ts,
                   batch_games_per_s=B / min(tb), seq_games_per_s=B / min(ts), speedup=min(ts) / min(tb),
                   batch_expanded_per_s=exp_b / min(tb), seq_expanded_per_s=exp_s / min(ts), expanded=exp_b,
                   batch_phase_ms=ph, e2e_solve_many_s=e2e_b, e2e_sequential_solve_s=e2e_s,
                   e2e_speedup=e2e_s / e2e_b, e2e_batch_games_per_s=B / e2e_b, e2e_seq_games_per_s=B / e2e_s,
                   e2e_batch_expanded_per_s=exp_e2e_b / e2e_b, e2e_seq_expanded_per_s=exp_e2e_s / e2e_s, moves=[len(m) - 1 for m in many], visited=batch_visited, parity=same)
        lines_out.append(rec)
        print(json.dumps(rec), flush=True)
        if not same:
            print('PARITY MISMATCH between State.solve_many and State.solve', file=sys.stderr)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            for r in lines_out:
                f.write(json.dumps(r) + '\n')
    return 0 if all(r.get('parity', True) for r in lines_out) else 1


if __name__ == '__main__':
    sys.exit(main())
