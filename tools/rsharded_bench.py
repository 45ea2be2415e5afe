"""Timing of realistic-mode solves on the key-sharded driver (RShardedSolver) and, on one rank, on the fused single-GPU
solver (spl_rsolver), under torchrun:
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 tools/rsharded_bench.py --beam 20000000
One JSON line per timed solve on rank 0 (and --out FILE collects them): ms per solve (CUDA events), expanded/s, a
digest of the per-level counters (frontier, generated, unique, kept: the same for every world size and for the fused
solver), the sha256 of every level's records in rank order when the beam is at most --record-digest-max, the visited
states per rank, and the device name and power limit."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch
import torch.distributed as dist

import splendor_rl_gym_b200 as S
from splendor_rl_gym_b200.sharded import Comm, RCudaBackend, RShardedSolver

ap = argparse.ArgumentParser()
ap.add_argument('--players', type=int, default=2)
ap.add_argument('--goal', type=int, default=15)
ap.add_argument('--seed', type=int, default=0, help='market shuffle seed (-1: unshuffled)')
ap.add_argument('--beam', type=int, default=20_000)
ap.add_argument('--steps', type=int, default=3)
ap.add_argument('--warmup', type=int, default=1)
ap.add_argument('--block-parents', type=int, default=1 << 20)
ap.add_argument('--fused', action='store_true', help='also time spl_rsolver (world size 1 only)')
ap.add_argument('--slots', type=int, default=0, help='initial realistic table buckets per rank (0: grow from the default)')
ap.add_argument('--max-table-gb', type=float, default=150.0)
ap.add_argument('--record-digest-max', type=int, default=1_000_000)
ap.add_argument('--out', default='')
ap.add_argument('--gloo', action='store_true',
                help='gloo process group with host-staged collectives, ranks sharing the visible GPUs round-robin '
                     '(checks N ranks on fewer than N GPUs; not a multi-GPU timing)')
a = ap.parse_args()

local = int(os.environ.get('LOCAL_RANK', '0')) % (torch.cuda.device_count() if a.gloo else 1 << 30)
torch.cuda.set_device(local)
if int(os.environ.get('WORLD_SIZE', '1')) > 1:
    if a.gloo:
        dist.init_process_group('gloo')
    else:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
eng = S.Engine(local, table_slots=a.slots, max_table_bytes=int(a.max_table_gb * 1e9))
comm = Comm(eng.tdev)
gpc = {2: 4, 3: 5, 4: 7}[a.players]
root = S.MultiPlayerState.newgame(S.GameConfig(num_players=a.players, target_points=a.goal, gems_per_color=gpc, infinite_resources=False),
                                  shuffle_market=a.seed >= 0, seed=a.seed if a.seed >= 0 else None)
rcfg = root.rconfig('const')


def device_line():
    try:
        q = subprocess.run(['nvidia-smi', f'--id={local}', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = repr(e)
    return q or torch.cuda.get_device_name(local)


def counters_digest(infos):
    h = hashlib.sha256()
    for i in infos:
        h.update(json.dumps([int(i[k]) for k in ('frontier', 'generated', 'unique', 'kept')]).encode())
    return h.hexdigest()


def solve(driver, digest):
    """one solve -> (infos, ms, per-level record digest or None, visited per rank)"""
    rec = hashlib.sha256() if digest else None
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    if driver == 'fused':
        sol = eng.rsolver(rcfg, root.record(), a.beam)
        while not sol.ended:
            sol.step()
            if rec is not None and not sol.ended:
                rec.update(sol.frontier().tobytes())
        infos = sol.infos
        sol.close()
        vis = [infos[-2]['visited'] if len(infos) > 1 else 1]
    else:
        sol = RShardedSolver(RCudaBackend(eng, rcfg, root.record()), comm, a.beam, block_parents=a.block_parents)
        while not sol.ended:
            gi = sol.step()
            if rec is not None and not gi['ended']:
                fr = sol.gather_frontier()
                if comm.rank == 0:
                    rec.update(fr.cpu().numpy().tobytes())
        infos = sol.infos
        vis = [int(x) for x in comm.gather_ints(sol.b.visited_count())[:, 0]]
    end.record()
    torch.cuda.synchronize()
    return infos, start.elapsed_time(end), (rec.hexdigest() if rec is not None else None), vis


lines = []
drivers = ['sharded'] + (['fused'] if a.fused and comm.world == 1 else [])
for driver in drivers:
    for step in range(a.warmup + a.steps):
        digest = step == a.warmup and a.beam <= a.record_digest_max  # the records' digest in an untimed extra pass
        infos, ms, _, vis = solve(driver, False)
        rec_digest = solve(driver, True)[2] if digest else None
        if step < a.warmup:
            continue
        expanded = sum(i['expanded'] for i in infos)
        line = dict(driver=driver, world=comm.world, players=a.players, goal=a.goal, seed=a.seed, beam=a.beam,
                    block_parents=a.block_parents if driver == 'sharded' else None, step=step - a.warmup,
                    ms_per_solve=round(ms, 3), levels=len(infos), expanded=expanded,
                    expanded_per_s=round(expanded / (ms / 1e3), 1), counters_digest=counters_digest(infos),
                    record_digest=rec_digest, visited_per_rank=vis, device=device_line() if comm.rank == 0 else None,
                    collectives=(f'gloo, host-staged, {comm.world} ranks on {torch.cuda.device_count()} GPU(s)' if a.gloo else 'nccl')
                    if comm.on else 'none')
        if comm.rank == 0:
            print(json.dumps(line), flush=True)
            lines.append(line)
if comm.rank == 0 and a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    with open(a.out, 'a') as f:
        for line in lines:
            f.write(json.dumps(line) + '\n')
if comm.on:
    dist.destroy_process_group()
