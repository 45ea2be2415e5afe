"""Formula heuristics on one GPU: what the formula path costs, and that the built-in path does not pay for it.

Measurements (one JSON line each, after a header line with the GPU's name and power limit, to stdout and to --out):
  ab        bench.py's default workload (C3: goal 15, `aggressive`, beam 30 M, noise const, stable ties) run by bench.py
            from a checkout of the parent commit with its library built (--parent-tree) and from this tree,
            alternating (parent first, then this tree first), --ab-reps runs each; bench.py's value and e2e per run, and
            whether every --dump-outputs array is identical between the two libraries
  twin      the same search through the API: the built-in `aggressive` against its formula twin
            (formula.BUILTIN_TWINS), alternating, --reps solves each: seconds per solve (host clock around work that ends
            in a device synchronise) and whether every level's counters and the line are identical
  sweep     64 formula variants of `aggressive` (coefficients and exponents varied), goal --sweep-goal, beam 300 000: one
            State.solve_many batch against the 64 State.solve calls in turn, once each after a warm-up; parity of the lines

    python tools/formula_bench.py --parent-tree ../parent-checkout --out profiles/fh1_formula_bench.jsonl
"""
import argparse
import hashlib
import json
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def gpu_header():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return {'gpu': q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None}


def run_bench(tree, dump_dir, steps, warmup):
    cmd = [sys.executable, str(Path(tree) / 'bench.py'), '--gpus', '1', '--steps', str(steps), '--warmup', str(warmup),
           '--no-cpu-baseline', '--no-parity', '--dump-outputs', dump_dir]
    p = subprocess.run(cmd, capture_output=True, text=True, cwd=tempfile.gettempdir())
    if p.returncode:
        raise RuntimeError(f'bench.py failed ({p.returncode}): {p.stderr[-2000:]}')
    line = [ln for ln in p.stdout.splitlines() if ln.startswith('{')][-1]
    return json.loads(line)


def dump_digest(d):
    import numpy as np
    return {f.name: hashlib.sha256(np.load(f).tobytes()).hexdigest() for f in sorted(Path(d).glob('*.npy'))}


def ab(a, out):
    rows = []
    for rep in range(a.ab_reps):
        order = [('parent', Path(a.parent_tree).resolve()), ('this', ROOT)]
        if rep % 2:
            order.reverse()
        for arm, tree in order:
            with tempfile.TemporaryDirectory() as d:
                r = run_bench(tree, d, a.steps, a.warmup)
                rows.append(dict(arm=arm, rep=rep, value=r['value'], e2e=r['e2e']['value'], dump=dump_digest(d)))
    per = {arm: [r for r in rows if r['arm'] == arm] for arm in ('parent', 'this')}
    same = all(r['dump'] == per['parent'][0]['dump'] for r in rows)
    out(dict(kind='ab', workload='bench.py C3 (goal 15, aggressive, beam 30 M)', steps=a.steps, warmup=a.warmup,
             runs=[{k: r[k] for k in ('arm', 'rep', 'value', 'e2e')} for r in rows],
             best_value={k: max(r['value'] for r in v) for k, v in per.items()},
             best_e2e={k: max(r['e2e'] for r in v) for k, v in per.items()},
             dump_outputs_identical=same, dump=per['this'][0]['dump']))


def solve_once(S, eng, h, goal, beam):
    import torch
    k, aux = S.State.newgame().record()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    sol = eng.solver(k, aux, goal, True, h, beam, 'stable', 'const')
    infos = sol.run()
    line = sol.path()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    sol.close()
    digest = hashlib.sha256(json.dumps([[i[f] for f in ('frontier', 'generated', 'unique', 'kept', 'visited')] for i in infos]
                                       + [line]).encode()).hexdigest()
    return dt, digest


def twin(a, out):
    import splendor_rl_gym_b200 as S
    from splendor_rl_gym_b200.formula import BUILTIN_TWINS
    eng = S.Engine.get(0)
    arms = {'builtin': 'aggressive', 'formula': BUILTIN_TWINS['aggressive']}
    for h in arms.values():
        solve_once(S, eng, h, 15, a.beam)  # warm-up: modules, pools, tables
    times, digests = {k: [] for k in arms}, {k: set() for k in arms}
    for rep in range(a.reps):
        names = list(arms) if rep % 2 == 0 else list(arms)[::-1]
        for n in names:
            dt, dg = solve_once(S, eng, arms[n], 15, a.beam)
            times[n].append(dt)
            digests[n].add(dg)
    out(dict(kind='twin', workload=f'goal 15, beam {a.beam}, noise const, stable ties', reps=a.reps,
             s_per_solve={k: v for k, v in times.items()}, best_s={k: min(v) for k, v in times.items()},
             median_s={k: sorted(v)[len(v) // 2] for k, v in times.items()},
             identical=len(digests['builtin'] | digests['formula']) == 1))


def sweep(a, out):
    import torch
    import splendor_rl_gym_b200 as S
    from splendor_rl_gym_b200 import Formula
    eng = S.Engine.get(0)
    variants = [Formula([(200.0 + 5 * (i % 8), ('pts', 3.0 + 0.05 * (i // 8))), (5.0, ('saved', 0.3)),
                         (2.0 + 0.25 * (i % 4), ('bonus', 0.5))]) for i in range(64)]
    roots = [S.State.newgame()] * len(variants)
    key = lambda line: [(s.cards, s.gems, s.pts, s.saved) for s in line]  # noqa: E731
    S.State.solve_many(roots[:2], a.sweep_goal, use_heuristic=True, heuristic_name=variants[:2], beam_width=a.sweep_beam)  # warm-up
    S.State.newgame().solve(a.sweep_goal, use_heuristic=True, heuristic_name=variants[0], beam_width=a.sweep_beam, verbose=False)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    batch = S.State.solve_many(roots, a.sweep_goal, use_heuristic=True, heuristic_name=variants, beam_width=a.sweep_beam)
    torch.cuda.synchronize()
    t_batch = time.perf_counter() - t0
    t0 = time.perf_counter()
    seq = [S.State.newgame().solve(a.sweep_goal, use_heuristic=True, heuristic_name=f, beam_width=a.sweep_beam, verbose=False)
           for f in variants]
    torch.cuda.synchronize()
    t_seq = time.perf_counter() - t0
    out(dict(kind='sweep', workload=f'64 formula variants of aggressive, goal {a.sweep_goal}, beam {a.sweep_beam}', games=len(variants),
             s_batch=t_batch, s_sequential=t_seq, speedup=t_seq / t_batch,
             lines_identical=all(key(x) == key(y) for x, y in zip(batch, seq)),
             distinct_lines=len({repr(key(x)) for x in batch})))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--parent-tree', default=None, help='checkout of the parent commit, library built (the ab measurement)')
    ap.add_argument('--ab-reps', type=int, default=2)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=1)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--beam', type=int, default=30_000_000)
    ap.add_argument('--sweep-beam', type=int, default=300_000)
    # goal 15 from the new game visits ~14 M states per game: 64 of them overflow the batch's visited table
    ap.add_argument('--sweep-goal', type=int, default=10)
    ap.add_argument('--only', default='ab,twin,sweep')
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    fh = open(a.out, 'a') if a.out else None

    def out(d):
        s = json.dumps(d)
        print(s, flush=True)
        if fh:
            fh.write(s + '\n')
            fh.flush()
    out(gpu_header())
    todo = a.only.split(',')
    if 'ab' in todo and a.parent_tree:
        ab(a, out)
    if 'twin' in todo:
        twin(a, out)
    if 'sweep' in todo:
        sweep(a, out)


if __name__ == '__main__':
    main()
