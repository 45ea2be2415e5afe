#!/usr/bin/env python
"""bench.py -- expanded states/sec of the frontier-expansion path (BASELINE.json's metric).

    python bench.py --gpus 1 --steps K --warmup W            # this repo's CUDA path
    python bench.py ... --dump-outputs DIR                   # ... and write what its last timed step computed (below)
    python bench.py --impl reference --steps K --warmup W    # the reference algorithm on host cores
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   # one rank per GPU

One "step" = one complete search (root -> first state with >= goal points): every level runs
generate + dedup + score + top-k.  Workloads (`--config`, all grown from the all-zero root state and the
rules' constant tables: synthetic by construction):
    C3 (default)  BASELINE configs[2]: speedrun goal 15, `aggressive`, beam 30 M per GPU (N GPUs: 30 M x N), noise
                  `const`, ties by arrival order (`stable`)
    C1            configs[0]: goal 10, `simple`, beam 300 000 (the reference's own CPU-runnable case)
    C4            configs[3]: goal 15, `balanced` (or --heuristic efficiency), beam 12.5 M per GPU (8 GPUs: 100 M); on N > 1 the
                  card-set-sharded driver reports more than 2048 distinct scores per level and the search reruns on the
                  key-sharded driver, as State.solve() does (named in config.parallelism)
    C2            configs[1]: exhaustive BFS to --bfs-depth levels (queue sharded by key hash on N > 1)
    C5            configs[4]: realistic mode, --players 2|3, goal 15, market seed 0, --beam 20000 | 2000000 (one GPU per
                  replica: realistic mode is not sharded)

    value         expanded states / s, timed on the device (CUDA events) over K solves whose state lives in HBM throughout
    e2e           the same metric through the public API (`State.newgame().solve(...)` / `MultiPlayerState...solve()`)
                  with host inputs/outputs: root record H2D, per-level counters and the winning line D2H, path replay
                  -- wall clock around the call; bytes as counted by the library and the Python layer
    roofline      dominant stage of the level (per-run dedup kernels of the card-set-grouped level): algorithmic bytes
                  / CUDA-event time; traffic = measured DRAM bytes per launch of those kernels
                  (profiles/dedup_stage_traffic.json, from the committed ncu launch list; N = 1, C3)
    parity_check  one untimed search at a CPU-feasible width through the SAME solver class, every level's queue
                  (records in rank order) hashed and compared with the CPU oracle's (rank 0 runs the oracle)
    cpu_baseline  the CPU oracle (C port of the reference algorithm, 1 thread) on a bounded sample of the same workload;
                  when the unmodified Python reference is staged under baseline/_ref/ it is timed in the same run too
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

R_BYTES, K_BYTES = 24, 16  # SURVEY.md 8(d): record = key + aux, key
RR_BYTES, RK_BYTES = 48, 32  # realistic mode
CPU_SAMPLE_BEAM = 300_000
PARITY_BEAM = 300_000
PER_GPU_BEAM = {'C3': 30_000_000, 'C4': 12_500_000}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--config', default='C3', choices=['C1', 'C2', 'C3', 'C4', 'C5'])
    ap.add_argument('--goal', type=int, default=None)
    ap.add_argument('--heuristic', default=None)
    ap.add_argument('--beam', type=int, default=None, help='total beam width (default: per-config, scaled by --gpus for C3/C4)')
    ap.add_argument('--noise', default='const')
    ap.add_argument('--tie', default='stable')
    ap.add_argument('--players', type=int, default=2)
    ap.add_argument('--bfs-depth', type=int, default=10)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-parity', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step computed to DIR/*.npy (float64), for comparing two builds')
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if a.dump_outputs and a.impl != 'b200':
        ap.error('--dump-outputs applies to the CUDA arm (--impl b200)')
    world = int(os.environ.get('WORLD_SIZE', '1'))
    d = {'C1': (10, 'simple', 300_000), 'C2': (255, 'simple', 0), 'C3': (15, 'aggressive', PER_GPU_BEAM['C3'] * world),
         'C4': (15, 'balanced', PER_GPU_BEAM['C4'] * world), 'C5': (15, 'competitive', 20_000)}[a.config]
    a.goal = a.goal if a.goal is not None else d[0]
    a.heuristic = a.heuristic or d[1]
    a.beam = a.beam if a.beam is not None else d[2]
    return a


# ------------------------------------------------------------------ clocks sampler
class ClockSampler:
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw'

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(',')]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 - 0.05 <= t <= t1 + 0.15 and len(r) >= 6] or [r for _, r in self.rows if len(r) >= 6]
        if not rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        sm = sorted(int(float(r[0])) for r in rows)
        reasons = [n for i, n in enumerate(['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'], 2)
                   if any(r[i].lower().startswith('active') for r in rows)]
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': int(float(rows[0][1])), 'reasons': reasons, 'samples': len(rows)}


# ------------------------------------------------------------------ CPU legs (oracle = C port of the reference algorithm)
def _level_hash(h, lo, hi, aux, link):
    import numpy as np
    rec = np.empty((len(lo), 4), dtype=np.uint64)
    rec[:, 0], rec[:, 1], rec[:, 2], rec[:, 3] = lo, hi, aux, link
    h.update(rec.tobytes())


def cpu_solve(a, beam, digest=False):
    """oracle search of the workload at width `beam` -> (expanded, seconds, levels, sha256 of every level's queue)"""
    import oracle
    h = hashlib.sha256()
    market = _market_seed0() if a.config == 'C5' else None  # (imports the package: outside the timed region)
    t0 = time.perf_counter()
    if a.config == 'C5':
        cfg = oracle.make_rconfig(a.players, a.goal, {2: 4, 3: 5, 4: 7}[a.players], market)
        s = oracle.RSolver(cfg, beam)
    else:
        s = oracle.Solver(a.goal, use_heuristic=a.config != 'C2', heuristic_name=a.heuristic, beam_width=beam, policy=a.tie, noise=a.noise)
    exp, levels = 0, 0
    while not s.done:
        info = s.step()
        if a.config == 'C2' and info['level'] + 1 >= beam_depth(a):
            s.done = True
        exp += info['expanded']
        levels += 1
        if digest and not s.done:
            if a.config == 'C5':
                h.update(s.level(info['level'] + 1).tobytes())
            else:
                st, lk = s.level(info['level'] + 1)
                _level_hash(h, st['lo'], st['hi'], st['aux'], lk)
    dt = time.perf_counter() - t0
    s.close()
    return exp, dt, levels, h.hexdigest()


def beam_depth(a):
    return min(a.bfs_depth, 8)  # BFS levels the CPU legs walk (level 8 -> 9 already takes minutes on one core)


def _market_seed0():
    """card market of `MultiPlayerState.newgame(cfg, shuffle_market=True, seed=0)` (src/solver.py:94-119): computed by
    this package's host mirror of CardMarket.from_full_deck with Python's own random.Random(0)"""
    import splendor_rl_gym_b200 as S
    m = S.CardMarket.from_full_deck(shuffle=True, seed=0)
    return [list(m.tier1_visible + m.tier1_deck), list(m.tier2_visible + m.tier2_deck), list(m.tier3_visible + m.tier3_deck)]


def python_reference_rate(a):
    """the unmodified Python reference (baseline/_ref, staged by build() from SPLENDOR_REFERENCE) on one core"""
    ref = ROOT / 'baseline' / '_ref'
    if a.config == 'C5' or a.config == 'C2' or not (ref / 'src' / 'solver.py').exists():
        return None
    beam = 2000
    try:
        out = subprocess.run([sys.executable, str(ROOT / 'tools' / 'ref_timing.py'), str(ref), str(a.goal), a.heuristic, str(beam)],
                             capture_output=True, text=True, timeout=300)
        r = json.loads(out.stdout.strip().splitlines()[-1])
        return {'value': r['expanded'] / r['seconds'], 'unit': 'expanded states/s', 'cores': 1, 'kind': 'reference',
                'sample': f"unmodified Python reference (baseline/_ref), goal {a.goal} {a.heuristic} beam {beam}, randint patched to 50: "
                          f"{r['expanded']} expanded in {r['seconds']:.1f} s, {r['moves']} moves"}
    except Exception as e:  # noqa: BLE001 -- a missing / broken staging must not break the bench line
        return {'unavailable': repr(e)[:200]}


def workload_name(a, world):
    if a.config == 'C5':
        return f'C5 (BASELINE configs[4]): realistic mode, {a.players} players, goal {a.goal}, market seed 0, beam {a.beam}, noise={a.noise}'
    if a.config == 'C2':
        return f'C2 (BASELINE configs[1]): exhaustive BFS from the root, {a.bfs_depth} levels'
    per = f' (= {a.beam // world} per GPU)' if world > 1 else ''
    return (f'{a.config} (BASELINE configs[{ {"C1": 0, "C3": 2, "C4": 3}[a.config] }]): speedrun goal {a.goal} -u -H {a.heuristic}, beam {a.beam}{per}, '
            f'noise={a.noise}, ties={a.tie}; one step = one full solve from the root state')


def run_reference(a):
    """`--impl reference`: the reference's algorithm on the host cores.  The reference is Python and its search loop is
    sequential by construction; the arm times the oracle's C port of it (1 thread) on a bounded sample of the workload,
    and reports the unmodified Python reference's own rate beside it when baseline/_ref is staged."""
    if int(os.environ.get('RANK', '0')) != 0:
        return
    beam = min(a.beam, CPU_SAMPLE_BEAM) if a.config != 'C2' else 0
    steps, warm = a.steps, min(a.warmup, 1)
    small = argparse.Namespace(**vars(a))
    for _ in range(warm):
        cpu_solve(small, min(beam, 20_000) if a.config != 'C2' else 0)
    exp = tot = 0.0
    for _ in range(steps):
        e, dt, _, _ = cpu_solve(a, beam)
        exp += e
        tot += dt
    v = exp / tot
    sample = f'{workload_name(a, 1)} -- bounded to beam {beam}' if a.config != 'C2' else f'BFS to depth {beam_depth(a)}'
    cb = {'value': v, 'unit': 'expanded states/s', 'cores': 1, 'kind': 'port', 'sample': sample, 'host_cores': os.cpu_count()}
    pr = python_reference_rate(a)
    if pr:
        cb['python_reference'] = pr
    print(json.dumps({
        'impl': 'reference', 'metric': 'expanded states/sec (gen+dedup+score+top-k)', 'value': v,
        'unit': 'expanded states/s', 'n_gpus': a.gpus, 'steps': steps, 'warmup': warm,
        'ms_per_step': tot / steps * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'u64 keys / f64 scores', 'data': 'synthetic',
        'config': {'workload': sample, 'note': 'CPU-bounded sample of the GPU arm\'s workload (same goal / heuristic / policy, narrower beam)'},
        'cpu_baseline': cb,
        'e2e': {'value': v, 'unit': 'expanded states/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }))


# ------------------------------------------------------------------ --dump-outputs
# DIR/levels.npy      [levels, 9]  per-level counters of the last timed solve, columns LEVEL_FIELDS (NaN: not reported)
# DIR/queue.npy       [rows, Wq]    its final queue (one GPU only): each record as Wq little-endian 32-bit words
#                                   (speedrun: lo, hi, aux, link -> Wq = 8; realistic mode: 96-byte records -> Wq = 24)
# DIR/queue_rows.npy  [rows]        queue rank of each dumped record: all of them, or a fixed seeded sample
# DIR/path.npy        [moves+1, Wp] the winning line of the last timed public-API solve (not C2), one state per row
#                                   (speedrun: State.record() as lo, hi, aux -> Wp = 6; realistic mode:
#                                   MultiPlayerState.record(), link all ones -> Wp = 24)
# Every value is an integer held exactly in float64.
LEVEL_FIELDS = ('level', 'ended', 'frontier', 'expanded', 'generated', 'unique', 'kept', 'goal_rank', 'visited')
QUEUE_DUMP_BYTES = 48 << 20  # queue sample + its row indices; the whole dump stays under 64 MB


def _words(rows_u8):
    import numpy as np
    return np.ascontiguousarray(rows_u8).view('<u4').astype(np.float64)


def level_array(infos):
    import numpy as np
    return np.array([[float(i.get(f, np.nan)) for f in LEVEL_FIELDS] for i in infos], dtype=np.float64).reshape(-1, len(LEVEL_FIELDS))


def queue_sample(sol, a, torch):
    """-> (queue ranks, record words) of a finished single-GPU solver's queue; above the QUEUE_DUMP_BYTES budget a
    sample of ranks drawn with seed 0, in queue order"""
    import numpy as np
    fr = sol.frontier()  # C5: host records [n]; otherwise a device int64 tensor [n, 4]
    n, rec_bytes = fr.shape[0], (96 if a.config == 'C5' else 32)
    cap = QUEUE_DUMP_BYTES // (8 * (rec_bytes // 4 + 1))
    rows = np.arange(n) if n <= cap else np.sort(np.random.default_rng(0).choice(n, cap, replace=False))
    if a.config == 'C5':
        raw = fr[rows].view(np.uint8)
    else:
        raw = fr[torch.from_numpy(rows).to(fr.device)].cpu().numpy().view(np.uint8)
    return rows.astype(np.float64), _words(raw.reshape(-1, rec_bytes))


def path_array(path, a):
    import numpy as np
    if a.config == 'C5':
        raw = np.concatenate([p.record() for p in path]).view(np.uint8)
    else:
        m64 = (1 << 64) - 1
        raw = np.array([(k & m64, k >> 64, aux) for k, aux in (p.record() for p in path)], dtype=np.uint64).view(np.uint8)
    return _words(raw.reshape(len(path), -1))


def dump_outputs(d, arrays):
    import numpy as np
    os.makedirs(d, exist_ok=True)
    for name, arr in arrays.items():
        np.save(os.path.join(d, name + '.npy'), arr)


# ------------------------------------------------------------------ GPU arm
class Runner:
    """one search of the workload on the device through the same solver classes the public API uses"""

    def __init__(self, a, S, eng, comm, torch):
        self.a, self.S, self.eng, self.comm, self.torch = a, S, eng, comm, torch
        self.k, self.aux = S.State.newgame().record()
        if a.config == 'C5':
            cfg = S.GameConfig(num_players=a.players, target_points=a.goal, gems_per_color={2: 4, 3: 5, 4: 7}[a.players], infinite_resources=False)
            self.root = S.MultiPlayerState.newgame(cfg, shuffle_market=True, seed=0)

    def solver(self, beam, keep_links=False):
        a, S, eng, comm = self.a, self.S, self.eng, self.comm
        if a.config == 'C5':
            return eng.rsolver(self.root.rconfig(a.noise), self.root.record(), beam, keep_links)
        if comm.world == 1:
            return eng.solver(self.k, self.aux, a.goal, a.config != 'C2', a.heuristic, beam, a.tie, a.noise, keep_links=keep_links)
        from splendor_rl_gym_b200.sharded import CudaBackend, GroupedShardedSolver, ShardedSolver
        if a.config != 'C2' and a.tie == 'stable' and a.noise == 'const' and not getattr(self, 'key_sharded', False):
            return GroupedShardedSolver(eng, comm, self.k, self.aux, a.goal, a.heuristic, beam, a.noise, keep_links=keep_links)
        return ShardedSolver(CudaBackend(eng), comm, self.k, self.aux, a.goal, a.config != 'C2', a.heuristic, beam, a.tie, a.noise, keep_links=keep_links)

    def run(self, beam, digest=False, keep=False):
        """-> (per-level infos, sha256 over every level's queue or None); keep=True leaves the finished solver open
        as self.kept (its final queue is read after the timed region; the caller closes it)"""
        if self.comm.world > 1 and not getattr(self, 'key_sharded', False):
            from splendor_rl_gym_b200.sharded import DictionaryOverflow
            try:
                return self._run(beam, digest, keep)
            except DictionaryOverflow:  # e.g. `balanced` at wide beams: as State.solve() does, rerun on the key-sharded driver
                self.key_sharded = True
        return self._run(beam, digest, keep)

    def _run(self, beam, digest=False, keep=False):
        a = self.a
        sol = self.solver(beam)
        h = hashlib.sha256() if digest else None
        infos = []
        try:
            while True:
                info = sol.step()
                infos.append(info)
                if a.config == 'C2' and not info['ended'] and len(infos) >= (beam_depth(a) if digest else a.bfs_depth):
                    break
                if info['ended']:
                    break
                if digest:
                    if a.config == 'C5':
                        h.update(sol.frontier().tobytes())
                    else:
                        fr = sol.gather_frontier() if self.comm.world > 1 else sol.frontier()
                        h.update(fr.cpu().numpy().tobytes())
        except BaseException:
            if hasattr(sol, 'close'):
                sol.close()
            raise
        if keep:
            self.kept = sol
        elif hasattr(sol, 'close'):
            sol.close()
        return infos, (h.hexdigest() if digest else None)


def run_b200(a):
    import torch
    import torch.distributed as dist

    import splendor_rl_gym_b200 as S
    from splendor_rl_gym_b200.sharded import Comm

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    replicas = a.config == 'C5' and world > 1  # realistic mode does not shard: N independent replicas
    # Visited set sized for the whole search up front so that the timed region never rehashes.  Beam search: card-set
    # node table (384 B per card set ever generated; ~1.55 sets per beam slot at goal 15).  BFS / realistic mode:
    # key table, three 20-byte slots per 64-byte bucket.
    per_gpu_beam = max(1, a.beam // (1 if replicas else world))
    if a.config == 'C2':
        eng = S.Engine(local, table_slots=int(min(3 << 30, 700_000_000 * 4.8 ** max(0, a.bfs_depth - 11) / world / 0.6)), max_table_bytes=int(150e9))
        table_note = 'key table'
    elif a.config == 'C5':
        eng = S.Engine(local, table_slots=int(min(3 << 30, max(1 << 22, a.beam * 300))), max_table_bytes=int(150e9))
        table_note = 'key table (identity fingerprints)'
    else:
        nodes = int(min(150e9 / 384, max(1 << 14, per_gpu_beam * 4)))
        eng = S.Engine(local, table_slots=1 << 22, node_slots=nodes, max_node_bytes=int(160e9))
        table_note = 'card-set node table %.1f GB per GPU' % (nodes * 384 / 1e9)
    comm = Comm(eng.tdev)
    if replicas:
        comm.on, comm.world, comm.rank = False, 1, 0
    runner = Runner(a, S, eng, comm, torch)

    # ---- parity: one untimed search at a CPU-feasible width through the same solver class, every level vs the oracle
    parity = None
    if not a.no_parity:
        pbeam = min(a.beam, PARITY_BEAM if a.config != 'C5' else 20_000)
        infos_p, dig = runner.run(pbeam, digest=True)
        if rank == 0:
            oexp, odt, olevels, odig = cpu_solve(a, pbeam, digest=True)
            gexp = sum(i['expanded'] for i in infos_p)
            parity = {'ok': bool(dig == odig and gexp == oexp), 'levels': len(infos_p), 'digest': dig[:32], 'oracle_digest': odig[:32],
                      'expanded': gexp, 'oracle_expanded': oexp,
                      'what': f'{"beam " + str(pbeam) if a.config != "C2" else "BFS depth " + str(beam_depth(a))}: sha256 over every level\'s queue '
                              f'(records in rank order) == CPU oracle\'s, through the same solver class as the timed run'}
            cpu_sample = (oexp, odt, pbeam)
        if world > 1:
            dist.barrier()

    for _ in range(a.warmup):
        infos = runner.run(a.beam)[0]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = eng.launch_count()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    ev0.record()
    all_infos = []
    for s in range(a.steps):
        all_infos.append(runner.run(a.beam, keep=bool(a.dump_outputs) and s == a.steps - 1)[0])
    ev1.record()
    torch.cuda.synchronize()
    t1 = time.time()
    if world > 1:
        dist.barrier()
    ms = ev0.elapsed_time(ev1)
    launches = eng.launch_count() - l0
    tm = torch.tensor([ms], dtype=torch.float64, device='cuda')
    # per-level counters of the sharded solvers are already global; replicas each did the whole work
    expanded = float(sum(i['expanded'] for inf in all_infos for i in inf)) * (world if replicas else 1)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        lt = torch.tensor([float(launches)], dtype=torch.float64, device='cuda')
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
        launches = int(lt.item())
    ms = float(tm.item())
    value = expanded / (ms * 1e-3)
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    outputs = {}
    if a.dump_outputs:  # the last timed solve: its per-level counters and, on one GPU, its final queue
        outputs['levels'] = level_array(all_infos[-1])
        if comm.world == 1:
            outputs['queue_rows'], outputs['queue'] = queue_sample(runner.kept, a, torch)
        if hasattr(runner.kept, 'close'):
            runner.kept.close()

    # ---- end to end through the public API (host inputs / outputs inside the timed region)
    def api_solve(stats):
        if a.config == 'C5':
            return runner.root.solve(beam_width=a.beam, verbose=False, noise=a.noise, engine=eng, stats=stats)
        if a.config == 'C2':  # exhaustive BFS never reaches a goal at these depths: the API call is the level stepper itself
            stats.extend(runner.run(a.beam)[0])
            return None
        return S.State.newgame().solve(goal_pts=a.goal, use_heuristic=True, heuristic_name=a.heuristic, beam_width=a.beam, verbose=False,
                                       tie_policy=a.tie, noise=a.noise, engine=eng, stats=stats)

    for _ in range(min(a.warmup, 3)):
        # untimed: the API path keeps parent links, whose per-level columns are allocated on first use
        # (e2e.seconds_each_solve_rank0 lists the timed solves one by one)
        api_solve([])
    h0, d0 = eng.transfer_bytes()
    st = []
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    te0 = time.perf_counter()
    per_solve = []
    for _ in range(a.steps):
        ts0 = time.perf_counter()
        path = api_solve(st)
        per_solve.append(round(time.perf_counter() - ts0, 4))
    torch.cuda.synchronize()
    te = time.perf_counter() - te0
    h1, d1 = eng.transfer_bytes()
    e2e_t = torch.tensor([te], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_exp = sum(i['expanded'] for i in st) * (world if replicas else 1)
    e2e = {'value': float(e2e_exp) / float(e2e_t.item()), 'unit': 'expanded states/s',
           'h2d_bytes_per_step': (h1 - h0) // a.steps, 'd2h_bytes_per_step': (d1 - d0) // a.steps,
           'bytes_note': 'rank 0, counted: library copies (spl_transfer_bytes) + the Python layer\'s path-replay tensors',
           'seconds_per_solve': float(e2e_t.item()) / a.steps, 'seconds_each_solve_rank0': per_solve}
    if a.config == 'C5' and path:
        e2e.update(plies=len(path) - 1, winner=path[-1].get_winner(), final_pts=[p.pts for p in path[-1].players])
    elif path:
        e2e.update(moves=len(path) - 1, final=repr(path[-1]), final_pts=path[-1].pts)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if a.dump_outputs:
        if path:  # the winning line the last timed API solve returned
            outputs['path'] = path_array(path, a)
        dump_outputs(a.dump_outputs, outputs)

    infos = all_infos[-1]
    lv = [i for i in infos if i['expanded'] and i.get('generated')]
    n = sum(i['expanded'] for i in lv)
    gen = sum(i['generated'] for i in lv)
    uniq = sum(i['unique'] for i in lv)
    kept = sum(i['kept'] for i in lv)
    peaks = {}
    try:
        peaks = json.load(open(ROOT / 'MEASURED_PEAKS.json'))
    except OSError:
        pass
    peak = float(peaks.get('hbm_gbs', 6650.0))
    peak_src = 'MEASURED_PEAKS.json hbm_gbs' if peaks else 'fallback 6650 GB/s (B200_PROFILING.md)'
    R, K = (RR_BYTES, RK_BYTES) if a.config == 'C5' else (R_BYTES, K_BYTES)
    share = 1.0 if (world == 1 or replicas) else 1.0 / world  # a rank of the sharded search does 1/N of the level
    # dedup stage: read each parent (R), one visited-set key lookup per candidate (K), one insert per new unique (R)
    stage_bytes = (R * n + K * gen + R * uniq) * share
    pipe_bytes = (R * n + K * gen + ((2 * R + 16) * uniq + 2 * R * kept if a.config != 'C2' else R * uniq)) * share
    if world > 1 and not replicas and 'ms_warp' in lv[0] and 'ms_thread' in lv[0]:  # card-set-sharded level (rank 0's stage times)
        ms_stage = {'sort': sum(i['ms_sort'] for i in lv), 'thread': sum(i['ms_thread'] for i in lv),
                    'warp': sum(i['ms_warp'] for i in lv), 'cta': sum(i['ms_cta'] for i in lv)}
        dedup_ms = ms_stage['thread'] + ms_stage['warp'] + ms_stage['cta']
        kernel = 'm2_group_tiny_kernel + m2_group_warp_kernel + m2_group_big_kernel (per-run dedup of the rank\'s card sets)'
        launches_k = 3 * len(lv)
    elif 'ms_expand' in (lv[0] if lv else {}):
        ms_stage = {s: sum(i['ms_' + s] for i in lv) for s in ('count', 'expand', 'resolve', 'select', 'sort')}
        ms_stage['warp_kernel'] = sum(i.get('ms_warp', 0.0) for i in lv)
        dedup_ms = ms_stage['expand']
        grouped = a.config in ('C1', 'C3', 'C4') and a.noise != 'mt'
        kernel = ('m2_group_tiny_kernel + m2_group_warp_kernel + m2_group_big_kernel (per-run dedup of the card-set-grouped level)'
                  if grouped else ('probe_list_kernel (realistic)' if a.config == 'C5' else 'expand_kernel<MODE_PROBE>'))
        chunk = (16 << 20) if grouped else (4 << 20)
        launches_k = max(1, sum(-(-i['frontier'] // chunk) for i in lv)) * (3 if grouped else 1)
    else:
        ms_stage, dedup_ms, kernel, launches_k = {}, 0.0, 'n/a', 1
    roofline = None
    if dedup_ms > 0:
        achieved = stage_bytes / (dedup_ms * 1e-3) / 1e9
        traffic = None
        prof = ROOT / 'profiles' / 'dedup_stage_traffic.json'
        if prof.exists() and a.config == 'C3' and world == 1:
            try:
                traffic = json.load(open(prof)).get('dram_bytes_per_launch')
            except (OSError, ValueError):
                traffic = None
        roofline = {'bound': 'hbm', 'kernel': kernel, 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                    'traffic': traffic, 'peak_source': peak_src,
                    'algorithmic_bytes': 'R*n + K*generated + R*unique with R=%d, K=%d (SURVEY.md 8d)%s' % (R, K, ', this rank\'s 1/N share' if share < 1 else ''),
                    'algorithmic_bytes_per_launch': stage_bytes / launches_k, 'avg_launch_ms': dedup_ms / launches_k, 'launches': launches_k,
                    'stage_ms': dedup_ms,
                    'pipeline_frac': (pipe_bytes / (ms / a.steps * 1e-3) / 1e9) / peak}
    line = {
        'metric': 'expanded states/sec (gen+dedup+score+top-k)', 'value': value, 'unit': 'expanded states/s',
        'n_gpus': world, 'steps': a.steps, 'warmup': a.warmup, 'ms_per_step': ms / a.steps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'u64 keys / f64 scores',
        'data': 'synthetic',
        'config': {'workload': workload_name(a, world),
                   'l2': f'working set ({table_note}) >> 126 MB L2; no flush needed',
                   'beam': a.beam, 'goal': a.goal, 'heuristic': a.heuristic,
                   'parallelism': (('single GPU, ' + ('card-set-grouped level' if a.config in ('C1', 'C3', 'C4') else 'key-table level')) if world == 1 else
                                   f'{world} independent replicas (realistic mode does not shard)' if replicas else
                                   f'queue sharded by key hash over {world} GPUs (key-sharded driver: candidates routed with NCCL all-to-all, radix-select beam cut; '
                                   f'the card-set-sharded driver was tried first and reported more than 2048 distinct scores per level)' if getattr(runner, 'key_sharded', False) else
                                   f'queue sharded by card set over {world} GPUs: gem takes local, card buys stored into their owner\'s '
                                   f'receive buffer over NVLink by the routing kernel (CUDA IPC peer mappings; SPL_NO_P2P=1: NCCL all-to-all), '
                                   f'merged-dictionary beam cut, sample-sort global ranks')},
        'time_to_solve_s': ms / a.steps * 1e-3,
        'generated_per_s': float(gen) * (world if replicas else 1) * a.steps / (ms * 1e-3) if gen else None,
        'levels': len(infos), 'expanded_per_step': n, 'generated_per_step': gen, 'unique_per_step': uniq,
        'visited': next((i['visited'] for i in reversed(infos) if i.get('visited')), None),
        'stage_ms_per_step': {k_: round(v, 3) for k_, v in ms_stage.items()},
        'roofline': roofline, 'e2e': e2e, 'gpu_launches': launches, 'clocks': clocks, 'parity_check': parity,
    }
    if not a.no_cpu_baseline and world == 1:
        if parity is not None and a.config != 'C2':
            cexp, cdt, cbeam = cpu_sample  # the oracle run of the parity check doubles as the timed CPU sample
        else:
            cbeam = min(a.beam, CPU_SAMPLE_BEAM)
            cexp, cdt, _, _ = cpu_solve(a, cbeam)
        cb = {'value': cexp / cdt, 'unit': 'expanded states/s', 'cores': 1, 'kind': 'port', 'host_cores': os.cpu_count(),
              'sample': f'oracle C port of the reference algorithm, {workload_name(a, 1)} bounded to '
                        f'{"beam " + str(cbeam) if a.config != "C2" else "depth " + str(beam_depth(a))} ({cexp} expanded in {cdt:.1f} s, incl. per-level digests)'}
        pr = python_reference_rate(a)
        if pr:
            cb['python_reference'] = pr
        line['cpu_baseline'] = cb
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    args = parse()
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)
